"""The drop-in boundary against the REAL reference, in this container (SURVEY 8b): every wrapper the reference's own Python
calls has the reference's signature (names, order, defaults), and the reference's `nerf/network_grid.py` + `nerf/renderer.py`
import and construct on top of OUR `gridencoder` / `raymarching` / `freqencoder` packages.  (Running them needs a GPU AND
the reference tree, which never coexist: /root/reference is absent on the GPU box - the GPU-side check is
tests/test_gpu_step_parity.py against oracle/ref_pipeline.py on the reference's own kernels.)"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from oracle.build_ref import REF  # noqa: E402  (the reference's source tree, NGP_REFERENCE_ROOT)

CODE = r'''
import argparse, importlib, inspect, os, sys, types
ROOT, REF = %r, %r
sys.path.insert(0, ROOT)
from oracle.make_golden_cpu import import_reference
import_reference()                                    # stubs for the absent optional deps of nerf/*.py
for name in [n for n in sys.modules if n.split(".")[0] in ("gridencoder", "raymarching", "freqencoder", "encoding", "activation", "nerf")]:
    del sys.modules[name]

def sigs(mod_rm, mod_grid, mod_freq):
    out = {}
    for fn in ("_near_far_from_aabb", "_sph_from_ray", "_morton3D", "_morton3D_invert", "_packbits", "_march_rays_train",
               "_composite_rays_train", "_march_rays", "_composite_rays"):
        out["raymarching." + fn] = str(inspect.signature(getattr(mod_rm, fn).forward))
    out["grid._grid_encode"] = str(inspect.signature(mod_grid._grid_encode.forward))
    out["GridEncoder.__init__"] = str(inspect.signature(mod_grid.GridEncoder.__init__))
    out["GridEncoder.forward"] = str(inspect.signature(mod_grid.GridEncoder.forward))
    out["FreqEncoder.__init__"] = str(inspect.signature(mod_freq.FreqEncoder.__init__))
    out["FreqEncoder.forward"] = str(inspect.signature(mod_freq.FreqEncoder.forward))
    return out

# --- the reference's own wrappers (its extension modules from oracle/_ref satisfy `import _raymarching` etc.)
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
sys.path.insert(0, REF)
import raymarching.raymarching as r_rm, gridencoder.grid as r_grid, freqencoder.freq as r_freq
ref = sigs(r_rm, r_grid, r_freq)
ref_public = sorted(n for n in dir(importlib.import_module("raymarching")) if not n.startswith("_"))
for name in [n for n in sys.modules if n.split(".")[0] in ("gridencoder", "raymarching", "freqencoder", "encoding", "activation")]:
    del sys.modules[name]
sys.path = [p for p in sys.path if p != REF and not p.endswith("oracle/_ref")]

# --- ours, ahead of the reference root: the reference's nerf/*.py now import OUR packages by their top-level names
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(ROOT, "single-stable-dreamfusion_b200"))
import raymarching.raymarching as m_rm, gridencoder.grid as m_grid, freqencoder.freq as m_freq
assert "single-stable-dreamfusion_b200" in m_rm.__file__
mine = sigs(m_rm, m_grid, m_freq)
bad = {k: (ref[k], mine[k]) for k in ref if ref[k] != mine[k]}
assert not bad, bad
mine_public = set(n for n in dir(importlib.import_module("raymarching")) if not n.startswith("_"))
missing = [n for n in ref_public if n not in mine_public and n not in ("torch", "time", "np", "Function", "custom_fwd", "custom_bwd", "nn")]
assert not missing, missing

import encoding                                        # the REFERENCE's factory (encoding.py:5-32) - it imports OUR encoders
assert encoding.__file__.startswith(REF)
from nerf.network_grid import NeRFNetwork as RefNet    # the REFERENCE's network + renderer classes ...
import nerf.renderer as ref_renderer
assert ref_renderer.__file__.startswith(REF) and ref_renderer.raymarching.__file__.startswith(os.path.join(ROOT, "single-stable"))
opt = argparse.Namespace(bound=1, cuda_ray=True, min_near=0.1, density_thresh=10, bg_radius=1.4)
net = RefNet(opt)                                      # ... construct on top of OUR GridEncoder / FreqEncoder
assert type(net.encoder).__module__ == "gridencoder.grid" and "single-stable-dreamfusion_b200" in sys.modules["gridencoder.grid"].__file__
assert type(net.encoder_bg).__module__ == "freqencoder.freq"
assert net.encoder.embeddings.shape == (903480, 2) and net.in_dim == 32 and net.in_dim_bg == 39
print("DROPIN_SURFACE_OK", len(ref))
''' % (ROOT, REF)


def test_reference_python_imports_and_constructs_on_the_dropin_packages():
    if not os.path.isdir(os.path.join(REF, "nerf")) or not os.path.isdir(os.path.join(ROOT, "oracle", "_ref")):
        pytest.skip("the reference tree / its built extension modules are not available here")
    out = subprocess.run([sys.executable, "-c", CODE], capture_output=True, text=True, timeout=600)
    assert "DROPIN_SURFACE_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-3000:])
