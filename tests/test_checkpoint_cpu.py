"""CPU tests of the checkpoint layout (SURVEY 8f-3): files in the reference Trainer's format (nerf/utils.py:847-968)
round-trip through the B200 model, and a reference-shaped state_dict loads by name."""
import argparse
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "single-stable-dreamfusion_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# the names a reference checkpoint of nerf/network_grid.NeRFNetwork (-O, bg_radius > 0) carries
REFERENCE_KEYS = ["aabb_train", "aabb_infer", "density_grid", "density_bitfield", "step_counter", "encoder.embeddings",
                  "encoder.offsets", "sigma_net.net.0.weight", "sigma_net.net.0.bias", "sigma_net.net.1.weight",
                  "sigma_net.net.1.bias", "sigma_net.net.2.weight", "sigma_net.net.2.bias", "bg_net.net.0.weight",
                  "bg_net.net.0.bias", "bg_net.net.1.weight", "bg_net.net.1.bias"]


def _model(seed):
    from ngp_b200.network_grid import NeRFNetwork
    torch.manual_seed(seed)
    return NeRFNetwork(argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4))


def test_state_dict_has_exactly_the_reference_names_and_shapes():
    sd = _model(0).state_dict()
    assert sorted(sd) == sorted(REFERENCE_KEYS)
    assert sd["encoder.embeddings"].shape == (903480, 2) and sd["encoder.offsets"].shape == (17,)
    assert sd["density_grid"].shape == (1, 128 ** 3) and sd["density_bitfield"].shape == (128 ** 3 // 8,)
    assert sd["density_bitfield"].dtype == torch.uint8 and sd["step_counter"].shape == (16, 2)
    assert sd["sigma_net.net.0.weight"].shape == (64, 32) and sd["sigma_net.net.2.weight"].shape == (4, 64)
    assert sd["bg_net.net.0.weight"].shape == (64, 39) and sd["bg_net.net.1.weight"].shape == (3, 64)


def test_checkpoint_roundtrip_in_the_reference_layout():
    from ngp_b200 import checkpoint as ck
    a, b = _model(0), _model(1)
    with torch.no_grad():
        a.density_grid.uniform_(0, 20)
        a.density_bitfield.random_(0, 255)
        a.step_counter.random_(0, 1000)
    a.mean_count, a.mean_density = 1234, 5.5
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "df_ep0007.pth")
        ck.save_checkpoint(path, a, epoch=7, global_step=700)
        raw = torch.load(path, weights_only=False)
        assert set(raw) == {"epoch", "global_step", "stats", "mean_count", "mean_density", "model"}
        info = ck.load_checkpoint(path, b)
    assert info["epoch"] == 7 and info["global_step"] == 700 and not info["missing_keys"] and not info["unexpected_keys"]
    assert b.mean_count == 1234 and b.mean_density == 5.5
    for (k, va), (_, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(va, vb), k


def test_reference_shaped_files_load():
    """A dict built the way the reference writes it (extra keys, 'best' files that are bare state_dicts)."""
    from ngp_b200 import checkpoint as ck
    a, b, c = _model(2), _model(3), _model(4)
    ref_file = {"epoch": 3, "global_step": 300, "stats": {"loss": [0.1]}, "mean_count": 77, "mean_density": 0.25,
                "model": dict(a.state_dict(), **{"ema_shadow.0": torch.zeros(1)}),      # an unexpected key is tolerated
                "optimizer": {"state": {}, "param_groups": []}, "lr_scheduler": {}, "scaler": {"scale": 65536.0}}
    info = ck.load_checkpoint(ref_file, b, model_only=True)
    assert info["unexpected_keys"] == ["ema_shadow.0"] and b.mean_count == 77
    assert torch.equal(b.encoder.embeddings, a.encoder.embeddings)
    ck.load_checkpoint(a.state_dict(), c)                                               # bare state_dict
    assert torch.equal(c.sigma_net.net[1].weight, a.sigma_net.net[1].weight)

    class _Opt:                                                                         # a foreign optimizer state is reported
        def load_state_dict(self, sd):
            raise RuntimeError("layout mismatch")
    info = ck.load_checkpoint(ref_file, b, optimizer=_Opt())
    assert info["epoch"] == 3 and any("optimizer" in w for w in info["warnings"])


def _manifest():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "ref_state_dict_manifest.json")) as f:
        return json.load(f)


def test_state_dict_matches_the_real_reference_models_manifest():
    """tests/golden/ref_state_dict_manifest.json = keys / shapes / dtypes of the REAL nerf/network_grid.NeRFNetwork's
    state_dict(), written by oracle/make_golden_host.py (which imports the reference); ours must be identical, key for
    key, in the same order of parameter groups."""
    man = _manifest()
    m = _model(0)
    sd = m.state_dict()
    assert sorted(sd) == sorted(man["keys"])
    for k, meta in man["keys"].items():
        assert list(sd[k].shape) == meta["shape"], k
        assert str(sd[k].dtype).replace("torch.", "") == meta["dtype"], k
    assert sum(p.numel() for p in m.parameters()) == man["n_parameters"]
    assert sd["encoder.offsets"].tolist() == man["offsets"]
    groups = [{"n_tensors": len(list(g["params"])), "lr_mult": g["lr"] / 1e-3} for g in m.get_params(1e-3)]
    assert groups == man["param_groups"]


def test_cross_load_with_the_real_reference_model():
    """With the reference's source tree present (NGP_REFERENCE_ROOT): build the REAL reference model, load its
    state_dict into ours and ours into it with strict=True, and round-trip a reference-Trainer-shaped checkpoint file."""
    import pytest
    from oracle.build_ref import REF
    if not os.path.isdir(os.path.join(REF, "nerf")) or not os.path.isdir(os.path.join(ROOT, "oracle", "_ref")):
        pytest.skip("the reference tree / its built extension modules are not available here")
    import subprocess
    code = r'''
import argparse, os, sys, tempfile, torch
ROOT = %r
sys.path.insert(0, ROOT)
from oracle.build_ref import REF
from oracle.make_golden_host import import_reference_grid_model
RefNet, _, _ = import_reference_grid_model()
opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
torch.manual_seed(1)
ref = RefNet(opt)
with torch.no_grad():
    ref.density_grid.uniform_(0, 20); ref.density_bitfield.random_(0, 255); ref.step_counter.random_(0, 1000)
ref_sd = {k: v.clone() for k, v in ref.state_dict().items()}
# the product package shadows the reference's top-level module names: import it in a clean module table
for name in [n for n in sys.modules if n.split(".")[0] in ("gridencoder", "raymarching", "freqencoder", "encoding", "activation", "nerf")]:
    del sys.modules[name]
sys.path = [p for p in sys.path if not p.startswith(REF) and not p.endswith("oracle/_ref")]
sys.path.insert(0, os.path.join(ROOT, "single-stable-dreamfusion_b200"))
from ngp_b200.network_grid import NeRFNetwork
from ngp_b200 import checkpoint as ck
torch.manual_seed(2)
mine = NeRFNetwork(opt)
res = mine.load_state_dict(ref_sd, strict=True)
for k, v in mine.state_dict().items():
    assert torch.equal(v, ref_sd[k]), k
torch.manual_seed(3)
mine2 = NeRFNetwork(opt)
ref.load_state_dict(mine2.state_dict(), strict=True)          # and the other way round
for k, v in ref.state_dict().items():
    assert torch.equal(v, mine2.state_dict()[k]), k
# a file as the reference Trainer writes it (nerf/utils.py:847-902)
state = {"epoch": 5, "global_step": 500, "stats": {"loss": [], "valid_loss": [], "results": [], "checkpoints": [], "best_result": None},
         "mean_count": 321, "mean_density": 1.25, "model": ref_sd}
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "df_ep0005.pth")
    torch.save(state, path)
    torch.manual_seed(4)
    mine3 = NeRFNetwork(opt)
    info = ck.load_checkpoint(path, mine3)
assert info["epoch"] == 5 and not info["missing_keys"] and not info["unexpected_keys"]
assert mine3.mean_count == 321 and mine3.mean_density == 1.25
assert torch.equal(mine3.encoder.embeddings, ref_sd["encoder.embeddings"])
print("CROSS_LOAD_OK")
''' % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert "CROSS_LOAD_OK" in out.stdout, out.stderr[-3000:]
