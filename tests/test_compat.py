"""CPU: the compat shim lets the UNMODIFIED reference networks import above our op boundary (no import-time JIT build)
and wires them to this package's ops.  The reference networks come from oracle/_ref/refpy (byte-compiled by build() when
the reference checkout is present) or from the checkout itself."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import build_ref, refimport

REFERENCE = build_ref.REFPY if build_ref.refpy_available() else refimport.REFERENCE_ROOT


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, "models")), reason="neither oracle/_ref/refpy nor the reference checkout present")
def test_reference_networks_import_through_the_shim():
    code = r'''
import sys
sys.path.insert(0, %r)
import torch.utils.cpp_extension as ext
def _no_jit(*a, **k): raise AssertionError("reference JIT build reached: shim not effective")
ext.load = _no_jit
import gangealing_b200.compat as compat
compat.install()
sys.path.insert(0, %r)
import torch
torch.Tensor.cuda = lambda self, *a, **k: self
from models.stylegan2 import networks
from models.spatial_transformers import warping_heads, spatial_transformer
import gangealing_b200.op as op
from gangealing_b200.stn import sampling
assert networks.upfirdn2d is op.upfirdn2d and networks.fused_leaky_relu is op.fused_leaky_relu
assert networks.FusedLeakyReLU is op.FusedLeakyReLU
assert warping_heads.MipmapWarp is sampling.MipmapWarp
g = networks.Generator(32, 32, 2)
stn = spatial_transformer.get_stn(["similarity", "flow"], flow_size=64, supersize=64)
assert isinstance(stn.stns[0].warp_head.warper, sampling.MipmapWarp)
from utils.splat2d_cuda import splat2d
from gangealing_b200.splat2d import splat2d as ours
assert splat2d is ours
try:
    g([torch.randn(1, 32)])
except RuntimeError as exc:
    assert "CUDA tensors only" in str(exc)      # the reference networks reached our (GPU-only) op boundary
else:
    raise AssertionError("expected the CUDA-only boundary to refuse CPU tensors")
print("shim ok")
''' % (ROOT, REFERENCE)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "shim ok" in res.stdout, res.stdout + res.stderr
