"""splat2d: CPU sanity of the restatement; GPU parity against the restatement AND the reference kernel itself
(oracle/_ref/libsplat_ref.so, compiled from the reference's splat_gpu_impl.cu by oracle/build_ref.py)."""
import math

import pytest
import torch

from conftest import Pinned, assert_close
from oracle import splat as SP

DEV = "cuda"


def _case(seed, n, p, c, h, w, sigma, spread=1.2):
    g = torch.Generator().manual_seed(seed)
    coords = torch.rand(n, p, 2, generator=g) * torch.tensor([w * spread, h * spread]) - torch.tensor([w, h]) * (spread - 1) / 2
    values = torch.randn(n, p, c, generator=g)
    inp = torch.randn(n, c, h, w, generator=g)
    sig = torch.full((n,), sigma)
    return inp, coords, values, sig


def test_oracle_single_point_footprint_and_weights():
    # one point at (x=2.25, y=3.5), sigma 0.5 -> footprint rows floor(2.5)..ceil(4.5), cols floor(1.25)..ceil(3.25)
    inp = torch.zeros(1, 2, 8, 8)
    coords = torch.tensor([[[2.25, 3.5]]])
    values = torch.tensor([[[2.0, -1.0]]])
    out, alpha, touched = SP.splat2d_ref(inp, coords, values, torch.tensor([0.5]), False, return_alpha=True)
    ys, xs = torch.nonzero(touched[0], as_tuple=True)
    assert (ys.min(), ys.max(), xs.min(), xs.max()) == (2, 5, 1, 4)
    a = math.exp(-((2 - 2.25) ** 2 + (3 - 3.5) ** 2) / (2 * 0.25))
    assert abs(alpha[0, 3, 2].item() - a) < 1e-6
    assert abs(out[0, 0, 3, 2].item() - 2.0) < 1e-5 and abs(out[0, 1, 3, 2].item() + 1.0) < 1e-5  # a*v/(a+1e-8)
    assert out[0, :, 0, 0].abs().max() == 0
    soft = SP.splat2d_ref(inp, coords, values, torch.tensor([0.5]), True)
    assert abs(soft[0, 0, 3, 2].item() - 2.0 * a) < 1e-6       # alpha < 1 is clamped to 1


def test_oracle_out_of_bounds_points_are_dropped():
    inp = torch.zeros(1, 1, 4, 4)
    coords = torch.tensor([[[4.0, 1.0], [-0.001, 1.0], [1.0, 4.0], [3.999, 3.999]]])  # x == W is dropped
    values = torch.ones(1, 4, 1)
    _, alpha, touched = SP.splat2d_ref(inp, coords, values, torch.tensor([0.3]), False, return_alpha=True)
    assert touched[0].sum() > 0 and touched[0, :2, :2].sum() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,c,h,w,sigma,soft", [(2, 500, 3, 32, 40, 0.7, False), (1, 2000, 3, 64, 64, 1.3, False),
                                                   (2, 300, 1, 48, 48, 0.3, True), (1, 100, 5, 16, 16, 1.0, False),
                                                   (1, 64, 9, 16, 16, 0.6, True), (3, 1, 3, 8, 8, 0.5, False)])
def test_splat2d_vs_oracle(n, p, c, h, w, sigma, soft):
    from gangealing_b200.splat2d import splat2d
    inp, coords, values, sig = _case(p + c, n, p, c, h, w, sigma)
    out = splat2d(inp.to(DEV), coords.to(DEV), values.to(DEV), sig.to(DEV), soft)
    ref, _, touched = SP.splat2d_ref(inp, coords, values, sig, soft, return_alpha=True)
    assert_close(out, ref, rtol=1e-4, what="splat2d")
    # index work: the set of touched pixels is exact (zero canvas -> nonzero exactly where a footprint landed)
    blank = torch.zeros(n, 1, h, w)
    ones = torch.ones(n, p, 1)
    hit = splat2d(blank.to(DEV), coords.to(DEV), ones.to(DEV), sig.to(DEV), False).cpu()[:, 0] > 0
    assert torch.equal(hit, touched)


@pytest.mark.gpu
def test_splat2d_duplicate_points_and_dense_mask():
    """contention cases: many identical points; a dense rasterised disc up-sampled 2x (config 4 style)."""
    from gangealing_b200.splat2d import splat2d
    h = w = 64
    pts = torch.tensor([[[10.3, 20.7]]]).repeat(1, 4096, 1)
    vals = torch.randn(1, 4096, 3, generator=torch.Generator().manual_seed(0))
    out = splat2d(torch.zeros(1, 3, h, w, device=DEV), pts.to(DEV), vals.to(DEV), torch.tensor([1.0], device=DEV), False)
    ref = SP.splat2d_ref(torch.zeros(1, 3, h, w), pts, vals, torch.tensor([1.0]), False)
    assert_close(out, ref, rtol=2e-4, what="duplicates")
    ys, xs = torch.meshgrid(torch.arange(128.), torch.arange(128.), indexing="ij")
    disc = ((ys - 64) ** 2 + (xs - 64) ** 2) < 40 ** 2
    pts = torch.stack([xs[disc] / 2 + 0.13, ys[disc] / 2 + 0.21], dim=1)[None]
    vals = torch.randn(1, pts.shape[1], 3, generator=torch.Generator().manual_seed(1))
    out = splat2d(torch.zeros(1, 3, h, w, device=DEV), pts.to(DEV), vals.to(DEV), torch.tensor([0.6], device=DEV), False)
    ref = SP.splat2d_ref(torch.zeros(1, 3, h, w), pts, vals, torch.tensor([0.6]), False)
    assert_close(out, ref, rtol=2e-4, what="dense disc")


@pytest.mark.gpu
def test_splat2d_against_the_reference_kernel():
    """Pins both the product kernel and the oracle to the reference's own CUDA kernel on identical inputs.  What the
    reference kernel computed is kept in tests/golden/reference_splat.npz (conftest.Pinned; GG_RECORD_GOLDEN=1 with
    oracle/_ref/ built recomputes it on the GPU)."""
    from gangealing_b200.splat2d import splat2d
    pin = Pinned("reference_splat")
    for n, p, c, h, w, sigma, soft in [(2, 800, 3, 40, 56, 0.9, False), (1, 5000, 3, 64, 64, 1.3, True)]:
        inp, coords, values, sig = _case(7 + p, n, p, c, h, w, sigma)
        d = [t.to(DEV).contiguous() for t in (inp, coords, values, sig)]

        def reference():
            from oracle import build_ref
            lib = build_ref.load_splat_ref()
            assert lib is not None, "oracle/_ref/libsplat_ref.so not built (python -m oracle.build_ref)"
            # host side of the reference, splat_gpu.c:20-41: zeros / clone / kernel / clamp / divide
            alpha = torch.zeros(n, h, w, device=DEV)
            acc = d[0].clone()
            lib.SplatForwardGpu(torch.cuda.current_stream().cuda_stream, d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(),
                                alpha.data_ptr(), acc.data_ptr(), p, c, h, w, n * p)
            torch.cuda.synchronize()
            a = alpha.view(n, 1, h, w)
            if soft:
                a = a.clamp(1.0)
            return acc / (a + 1e-8), acc / (a + 1e-8), (alpha > 0).float()
        got = (splat2d(d[0], d[1], d[2], d[3], soft), SP.splat2d_ref(inp, coords, values, sig, soft),
               SP.splat2d_ref(inp, coords, values, sig, soft, return_alpha=True)[2].float())
        (ours, ref_out), (oracle, ref_out2) = pin("case%d" % p, got[:2], lambda: reference()[:2])
        covered, ref_covered = pin("covered%d" % p, got[2], lambda: reference()[2], keep=n * h * w)
        assert_close(ours, ref_out, rtol=1e-4, what="vs reference kernel")
        assert_close(oracle, ref_out2, rtol=1e-4, what="oracle vs reference kernel")
        assert torch.equal(covered, ref_covered)  # same pixel set
    pin.save()


@pytest.mark.gpu
def test_splat2d_argument_checks_and_call_site_contract():
    from gangealing_b200.splat2d import Splat2D, splat2d
    inp, coords, values, sig = _case(3, 2, 50, 3, 16, 16, 0.7)
    with pytest.raises(NotImplementedError):
        splat2d(inp, coords, values, sig, False)                       # CPU tensors: same error type as the reference
    with pytest.raises(AssertionError):
        splat2d(inp.to(DEV), coords[:1].to(DEV), values.to(DEV), sig.to(DEV), False)
    out = splat2d(inp.to(DEV).requires_grad_(True), coords.to(DEV), values.to(DEV), sig.to(DEV), False)
    with pytest.raises(NotImplementedError):
        out.sum().backward()                                           # forward only, like the reference
    # splat_points contract (utils/vis_tools/helpers.py:178-187)
    imgs = torch.rand(2, 3, 16, 16) * 2 - 1
    colors = torch.randn(2, 50, 3)
    pts = torch.rand(2, 50, 2) * 15
    expect = SP.splat_points_ref(imgs, pts, 0.7, 0.75, colors)
    got = SP.splat_points_ref(imgs.to(DEV), pts.to(DEV), 0.7, 0.75, colors.to(DEV), splat_fn=Splat2D())
    assert_close(got, expect, rtol=2e-4, what="splat_points")


# ------------------------------------------------------------------------------------------------ point-transfer kernels
@pytest.mark.gpu
def test_nn_argmin_kernel_against_the_reference_formulation():
    """congeal_points' brute-force search (spatial_transformer.py:655-668): the tiled argmin kernel against the reference's
    expanded-distance tensor + argmin on the CPU -- EXACT indices wherever the two smallest distances are separated."""
    from gangealing_b200.splat2d import nn_argmin
    g = torch.Generator().manual_seed(8)
    for n, h, w, p in [(2, 16, 16, 37), (1, 128, 128, 3000), (3, 24, 40, 1)]:
        ys, xs = torch.meshgrid(torch.linspace(-1, 1, h), torch.linspace(-1, 1, w), indexing="ij")
        grid = torch.stack([xs, ys], -1)[None].repeat(n, 1, 1, 1) + 0.05 * torch.randn(n, h, w, 2, generator=g)
        pts = torch.rand(n, p, 2, generator=g) * 2 - 1
        gg_ = grid.reshape(n, h, w, 1, 1, 2)
        pp = pts.reshape(n, 1, 1, p, 2, 1)
        sim = (gg_ @ pp)[..., 0, 0]
        dist = (pp.pow(2).squeeze(-1).sum(dim=-1) + gg_.pow(2).sum(dim=-1).squeeze(-1) - 2 * sim).reshape(n, h * w, p)
        expect = dist.argmin(dim=1)
        got = nn_argmin(grid.to(DEV), pts.to(DEV)).cpu()
        top2 = dist.topk(2, dim=1, largest=False).values
        decided = (top2[:, 1] - top2[:, 0]) > 1e-6
        assert decided.float().mean() > 0.95
        assert torch.equal(got[decided], expect[decided])
        # wherever the kernel disagrees on an undecided pair it still picked a (numerically) minimal entry
        picked = dist.gather(1, got[:, None, :]).squeeze(1)
        assert torch.all(picked <= top2[:, 0] + 1e-5)
    # exact duplicates: the first index wins, like argmin
    grid = torch.zeros(1, 4, 4, 2)
    assert int(nn_argmin(grid.to(DEV), torch.zeros(1, 1, 2, device=DEV))) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [0.3, 1.3])
def test_splat2d_lookup_fuses_uncongeal_points_into_the_splat(sigma):
    """`uncongeal_points` (grid_sample of the sampling grid at the query points + unnormalize, spatial_transformer.py:141-157)
    fused into the splat's point load: looked-up points and the splatted image against the two-step CPU oracle."""
    import torch.nn.functional as F
    from gangealing_b200.splat2d import splat2d_lookup
    g = torch.Generator().manual_seed(12)
    n, h, p, res = 2, 64, 5000, 64
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, 32), torch.linspace(-1, 1, 32), indexing="ij")
    grid = torch.stack([xs, ys], -1)[None].repeat(n, 1, 1, 1) * 0.9 + 0.03 * torch.randn(n, 32, 32, 2, generator=g)
    query = torch.rand(n, p, 2, generator=g) * 2.2 - 1.1          # some queries beyond the border
    vals = torch.randn(n, p, 3, generator=g)
    sig = torch.full((n,), sigma)
    looked = F.grid_sample(grid.permute(0, 3, 1, 2), query.unsqueeze(2), padding_mode="border", align_corners=False)
    looked = looked.squeeze(3).permute(0, 2, 1)
    pts = looked.div((res - 1) / res).div(2).add(0.5).mul(res - 1)            # SpatialTransformer.unnormalize
    expect = SP.splat2d_ref(torch.zeros(n, 3, h, h), pts, vals, sig, False)
    out, got_pts = splat2d_lookup(torch.zeros(n, 3, h, h, device=DEV), grid.to(DEV), query.to(DEV), vals.to(DEV), sig.to(DEV),
                                  res, res, False)
    assert_close(got_pts, pts, atol=2e-4, what="looked-up points (pixels)")
    assert_close(out, expect, rtol=2e-3, what="splatted image")
