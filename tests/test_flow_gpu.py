"""GPU parity of the fused flow composition (csrc/flow.cu)."""
import pytest
import torch

from conftest import assert_close, golden_cases, load_golden
from oracle import flow as FL

pytestmark = pytest.mark.gpu
DEV = "cuda"


def test_flow_compose_golden_forward_backward():
    from gangealing_b200 import stn
    blob = load_golden("flow_compose")
    for name in [n for n in golden_cases(blob) if n.startswith("case")]:
        s = int(blob[name + ".s"])
        low, mask, base = [blob[name + k].to(DEV).requires_grad_(True) for k in (".low", ".mask", ".base")]
        ident = FL.identity_flow_ref(s * low.shape[1], s * low.shape[2]).to(DEV)
        delta, flow = stn.flow_compose(low, mask, ident, base, None, s)
        assert_close(delta, blob[name + ".delta"], rtol=1e-5, what=name + " delta")
        assert_close(flow, blob[name + ".flow"], rtol=1e-5, what=name + " flow")
        grads = torch.autograd.grad((delta * blob[name + ".gd"].to(DEV)).sum() + (flow * blob[name + ".gf"].to(DEV)).sum(),
                                    [low, mask, base])
        for g, k in zip(grads, (".g_low", ".g_mask", ".g_base")):
            assert_close(g, blob[name + k], rtol=2e-4, what=name + k)
        up = stn.upsample_flow(low.detach(), mask.detach(), s)
        assert_close(up, blob[name + ".delta"], rtol=1e-5, what=name + " upsample_flow")


@pytest.mark.parametrize("n,with_base,with_alpha", [(5, True, False), (3, False, False), (4, True, True)])
def test_flow_compose_training_shape_vs_oracle(n, with_base, with_alpha):
    from gangealing_b200 import stn
    g = torch.Generator().manual_seed(n)
    low = 0.03 * torch.randn(n, 16, 16, 2, generator=g)
    mask = torch.randn(n, 576, 16, 16, generator=g)
    base = (torch.eye(2, 3)[None] + 0.1 * torch.randn(n, 2, 3, generator=g)) if with_base else None
    alpha = torch.rand(n, generator=g) if with_alpha else None
    ident = FL.identity_flow_ref(128, 128)
    leaves_o = [t.clone().requires_grad_(True) for t in (low, mask)] + ([base.clone().requires_grad_(True)] if with_base else [])
    d_o, f_o = FL.flow_compose_ref(leaves_o[0], leaves_o[1], ident, leaves_o[2] if with_base else None, alpha, 8)
    gd, gf = torch.randn(d_o.shape, generator=g), torch.randn(f_o.shape, generator=g)
    grads_o = torch.autograd.grad((d_o * gd).sum() + (f_o * gf).sum(), leaves_o)
    leaves = [t.to(DEV).requires_grad_(True) for t in (low, mask)] + ([base.to(DEV).requires_grad_(True)] if with_base else [])
    d, f = stn.flow_compose(leaves[0], leaves[1], ident.to(DEV), leaves[2] if with_base else None,
                            None if alpha is None else alpha.to(DEV), 8)
    assert_close(d, d_o, rtol=1e-5, what="delta")
    assert_close(f, f_o, rtol=1e-5, what="flow")
    grads = torch.autograd.grad((d * gd.to(DEV)).sum() + (f * gf.to(DEV)).sum(), leaves)
    for a, e, nm in zip(grads, grads_o, ("low", "mask", "base")):
        assert_close(a, e, rtol=3e-4, what="grad " + nm)


def test_apply_affine_drop_in():
    from gangealing_b200 import stn
    g = torch.Generator().manual_seed(0)
    m = torch.randn(3, 2, 3, generator=g)
    grid = torch.randn(3, 9, 7, 2, generator=g)
    assert_close(stn.apply_affine(m.to(DEV), grid.to(DEV)), FL.apply_affine_ref(m, grid), rtol=1e-5)


def test_flow_sampler_backward_is_reproducible_at_the_training_shape():
    """The flow STN's sampling backward (grid gradient with the level-of-detail term, flow composition: low-res flow, mask,
    similarity warp) sums in a fixed order: the same inputs give the same bits on every call, at the benchmark's shapes
    (per-GPU batch 32, 256^2 source, 128^2 flow from 16^2 cells)."""
    from gangealing_b200.stn import sampling as S
    g = torch.Generator().manual_seed(3)
    n = 32
    img = (torch.rand(n, 3, 256, 256, generator=g) * 2 - 1).to(DEV)
    low = (0.03 * torch.randn(n, 16, 16, 2, generator=g)).to(DEV)
    mask = torch.randn(n, 576, 16, 16, generator=g).to(DEV)
    theta = (torch.eye(2, 3)[None] * (0.6 + 0.8 * torch.rand(n, 1, 1, generator=g)) + 0.1 * torch.randn(n, 2, 3, generator=g)).to(DEV)
    ident = FL.identity_flow_ref(128, 128).to(DEV)
    go = torch.randn(n, 3, 128, 128, generator=g).to(DEV)

    def grads():
        leaves = [t.clone().requires_grad_(True) for t in (low, mask, theta)]
        out = S.stn_sample_flow(img, leaves[0], leaves[1], ident, leaves[2], None, 8, 3.5, 0.0, "reflection")[0]
        return torch.autograd.grad(out, leaves, go)
    first = grads()
    assert all(t.abs().max() > 0 for t in first)
    for _ in range(3):
        assert all(torch.equal(a, b) for a, b in zip(first, grads()))
