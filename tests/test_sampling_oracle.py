"""CPU: the sampler restatement (explicit index arithmetic) reproduces the reference-generated fixtures, and its
autograd gradient is the derivative of what it computes."""
import pytest
import torch

from conftest import assert_close, golden_cases, load_golden
from oracle import sampling as S


def test_mipmap_warp_oracle_matches_reference_fixtures():
    blob = load_golden("mipmap_warp")
    names = golden_cases(blob)
    assert len(names) >= 8
    for name in names:
        mode = S.PAD_MODES[int(blob[name + ".mode"])]
        x = blob[name + ".x"].clone().requires_grad_(True)
        grid = blob[name + ".grid"].clone().requires_grad_(True)
        y, aux = S.mipmap_warp_ref(x, grid, 3.5, 0.0, mode, return_aux=True)
        assert_close(y, blob[name + ".y"], rtol=5e-6, what=name)
        gx, gg = torch.autograd.grad(y, [x, grid], blob[name + ".go"])
        assert_close(gx, blob[name + ".gx"], rtol=2e-5, what=name + " gx")
        assert_close(gg, blob[name + ".ggrid"], rtol=2e-4, what=name + " ggrid")
        assert_close(aux["levels"], blob[name + ".levels"], rtol=1e-6, what=name + " levels")
        assert_close(S.warp_ref(blob[name + ".x"], blob[name + ".grid"], mode), blob[name + ".warp_y"], rtol=5e-6)


def test_level_indices_are_integers_in_range():
    blob = load_golden("mipmap_warp")
    for name in golden_cases(blob):
        _, aux = S.mipmap_warp_ref(blob[name + ".x"], blob[name + ".grid"], 3.5, 0.0, "border", return_aux=True)
        assert aux["level_0"].min() >= 0 and aux["level_1"].max() <= 3
        assert aux["num_levels"] == int(aux["level_1"].max()) + 1


def test_bilinear_downsample_oracle():
    blob = load_golden("bilinear_downsample")
    for stride in (2, 4):
        assert_close(S.bilinear_downsample_ref(blob["x"], stride), blob["s%d.y" % stride], rtol=1e-6)


def _smooth_field(n, h, w, gen, cells=6):
    """A smooth random displacement field (N, h, w, 2): bicubic up-sampling of a cells x cells random grid."""
    import torch.nn.functional as F
    coarse = torch.randn(n, 2, cells, cells, generator=gen, dtype=torch.float64)
    return F.interpolate(coarse, size=(h, w), mode="bicubic", align_corners=False).permute(0, 2, 3, 1)


@pytest.mark.parametrize("mode", S.PAD_MODES)
def test_oracle_grid_gradient_matches_finite_differences(mode):
    """The float64 oracle's autograd grid gradient (what the GPU sampler's backward is judged by) equals central finite
    differences of the loss, on the pixels where the gradient is decided (S.decided_pixels); the mask must keep nearly
    all of them.  The grid reaches the zeros / clip / fold regions of each padding mode and both level clamps."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(11 + S.PAD_MODES.index(mode))
    n, hs, ws, ho, wo = 3, 32, 32, 16, 12
    x = torch.randn(n, 3, hs, ws, generator=g, dtype=torch.float64)
    theta = torch.tensor([[[0.3, 0.05, 0.1], [-0.04, 0.35, -0.05]], [[1.3, 0.25, 0.1], [-0.2, 0.9, -0.05]],
                          [[3.4, -0.4, 0.3], [0.5, 2.8, 0.2]]], dtype=torch.float64)
    grid = F.affine_grid(theta, (n, 3, ho, wo), align_corners=False) + 0.04 * _smooth_field(n, ho, wo, g)
    go = torch.randn(n, 3, ho, wo, generator=g, dtype=torch.float64)
    levels = S.mipmap_levels(grid, hs, ws, 3.5)
    assert (levels == 0).any() and (levels == 2.5).any() and ((levels > 0) & (levels < 2.5)).any()

    def loss_map(gr):      # per output pixel
        return (S.mipmap_warp_ref(x, gr, 3.5, 0.0, mode) * go).sum(dim=1)
    gr = grid.clone().requires_grad_(True)
    (auto,) = torch.autograd.grad(loss_map(gr).sum(), gr)
    # A grid point enters the loss of its own pixel and of its four neighbours (their level of detail).  Points of one
    # colour (x + 2y) mod 5 are more than 2 apart, so no pixel sees two of them: one pair of evaluations per colour
    # and component gives every point's difference quotient, summed over the pixels it reaches.
    h = 1e-7
    ys, xs = torch.meshgrid(torch.arange(ho), torch.arange(wo), indexing="ij")
    colour = (xs + 2 * ys) % 5
    fd = torch.empty_like(grid)
    for c in range(5):
        for comp in range(2):
            e = torch.zeros_like(grid)
            e[:, colour == c, comp] = h
            d = F.pad((loss_map(grid + e) - loss_map(grid - e)) / (2 * h), (1, 1, 1, 1))
            reach = d[:, 1:-1, 1:-1] + d[:, 1:-1, :-2] + d[:, 1:-1, 2:] + d[:, :-2, 1:-1] + d[:, 2:, 1:-1]
            fd[:, colour == c, comp] = reach[:, colour == c]
    ok = S.decided_pixels(grid, hs, ws, mode, 3.5)
    assert ok.double().mean() >= 0.9
    err = (fd - auto)[ok].abs().max().item()
    print("fd %s: decided %.4f, max err %.2e of %.2e" % (mode, ok.double().mean().item(), err, auto.abs().max().item()))
    assert err <= 1e-6 * auto.abs().max().item(), "max err %.3e (grad magnitude %.3e)" % (err, auto.abs().max().item())


def test_oracle_theta_gradient_matches_finite_differences():
    """d loss / d theta of the float64 oracle (affine_grid_ref -> mipmap_warp_ref) equals central finite differences
    for an anisotropic affine warp.  Output pixels whose gradient is not decided are left out of the loss (a zero
    cotangent), so that no step crosses a kink; on an affine grid a left/right or up/down tie is decided for theta."""
    g = torch.Generator().manual_seed(5)
    n, hs, ws, ho, wo = 2, 64, 64, 20, 24
    x = torch.randn(n, 3, hs, ws, generator=g, dtype=torch.float64)
    theta = torch.tensor([[[1.73, 0.31, 0.07], [-0.22, 1.18, -0.11]], [[0.61, -0.13, 0.04], [0.27, 2.34, 0.09]]],
                         dtype=torch.float64)
    grid = S.affine_grid_ref(theta, (n, 3, ho, wo))
    ok = S.decided_pixels(grid, hs, ws, "border", 3.5, axis_ties=True)
    assert ok.double().mean() >= 0.9
    go = torch.randn(n, 3, ho, wo, generator=g, dtype=torch.float64) * ok[:, None]

    def loss(t):
        return (S.mipmap_warp_ref(x, S.affine_grid_ref(t, (n, 3, ho, wo)), 3.5, 0.0, "border") * go).sum()
    th = theta.clone().requires_grad_(True)
    (auto,) = torch.autograd.grad(loss(th), th)
    h = 1e-7
    fd = torch.empty_like(theta)
    for i in range(theta.numel()):
        e = torch.zeros(theta.numel(), dtype=torch.float64)
        e[i] = h
        fd.view(-1)[i] = (loss(theta + e.reshape(theta.shape)) - loss(theta - e.reshape(theta.shape))) / (2 * h)
    err = (fd - auto).abs().max().item()
    print("fd theta: decided %.4f, max err %.2e of %.2e" % (ok.double().mean().item(), err, auto.abs().max().item()))
    assert err <= 1e-6 * auto.abs().max().item(), "max err %.3e (grad magnitude %.3e)" % (err, auto.abs().max().item())


def test_affine_grid_restatement():
    import torch.nn.functional as F
    theta = torch.tensor([[[1.2, -0.3, 0.1], [0.3, 1.2, -0.2]]])
    assert_close(S.affine_grid_ref(theta, (1, 3, 5, 7)), F.affine_grid(theta, (1, 3, 5, 7), align_corners=False), rtol=1e-6)
