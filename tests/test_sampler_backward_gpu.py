"""GPU: the backward of the STN's sampler (csrc/warp.cu) and of the flow composition (csrc/flow.cu) against a float64
oracle (oracle/sampling.py, oracle/flow.py, run with autograd on the CPU).

The oracle is fed exactly what the kernel saw: the fp32 grid (or the grid the fused forward returned) cast up, and half
precision images and output gradients rounded to their type first.  The sampler's gradient is only piecewise smooth,
so per-pixel grid gradients are compared on the pixels where it is decided (oracle.sampling.decided_pixels), on
perturbed grids, and the decided fraction is asserted so that the mask cannot hide a bug.  Reductions over pixels (the
head parameters' gradients) are judged against the sum of the absolute per-pixel contributions, plus what the
undecided pixels could contribute.  The fused paths must equal, bit for bit, the separate kernels they are made of."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import flow as FL
from oracle import sampling as S

pytestmark = pytest.mark.gpu
DEV = "cuda"
LEVELS = 3.5                 # MipmapWarp(3.5): levels 0 .. 2.5, as the golden fixtures use
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
EPS = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}   # rounding of a returned half value
MIN_DECIDED = 0.98


def _smp():
    from gangealing_b200.stn import sampling
    return sampling


def _stn():
    from gangealing_b200 import stn
    return stn


def _report(what, **values):
    print("[%s] %s" % (what, ", ".join("%s %.3g" % kv for kv in values.items())))


def _random_thetas(n, hs, ws, ho, wo, gen, spacings=None):
    """(N, 2, 3) float64 anisotropic affine matrices: rotation x unequal axis scales + shear + shift.  Sample i puts
    neighbouring output pixels about spacings[i] source pixels apart (the level of detail is log2 of that); by default
    the spacings cycle through zoom-in (level clamped at 0), between, and beyond the last level (clamped at max)."""
    r = max((ws - 1.0) / wo if wo > 1 else 0.0, (hs - 1.0) / ho if ho > 1 else 0.0)
    if spacings is None:
        spacings = [(0.6, 2.4, 9.0)[i % 3] for i in range(n)]
    out = []
    for sp in spacings:
        u = torch.rand(5, generator=gen, dtype=torch.float64)
        a = 2 * math.pi * u[0].item()
        ani = 0.15 + 0.15 * u[1].item()
        s = sp / r
        rot = torch.tensor([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]], dtype=torch.float64)
        lin = rot @ torch.tensor([[s * (1 + ani), s * 0.1 * (u[2].item() - 0.5)], [0.0, s * (1 - ani)]], dtype=torch.float64)
        shift = 0.2 * (u[3:5] - 0.5).reshape(2, 1)
        out.append(torch.cat([lin, shift], dim=1))
    return torch.stack(out)


def _smooth_field(n, h, w, gen, cells=16):
    coarse = torch.randn(n, 2, cells, cells, generator=gen, dtype=torch.float64)
    return F.interpolate(coarse, size=(h, w), mode="bicubic", align_corners=False).permute(0, 2, 3, 1)


def _perturbed_grid(n, hs, ws, ho, wo, gen):
    """Affine (_random_thetas) plus a smooth random field of a few source pixels, fp32 (N, Ho, Wo, 2): no exact ties
    between neighbour distances, levels spread over the whole range, pixels outside the source."""
    theta = _random_thetas(n, hs, ws, ho, wo, gen)
    amp = 3.0 / max(hs, ws)
    return (F.affine_grid(theta, (n, 1, ho, wo), align_corners=False) + amp * _smooth_field(n, ho, wo, gen)).float()


def _oracle_warp(x64, grid64, go64, mip, min_level, mode, need_x=True):
    """float64 oracle: (out, d out.go / d x, d out.go / d grid)."""
    xl = x64.clone().requires_grad_(need_x)
    gl = grid64.clone().requires_grad_(True)
    out = S.mipmap_warp_ref(xl, gl, LEVELS, min_level, mode) if mip else S.warp_ref(xl, gl, mode)
    grads = torch.autograd.grad(out, [xl, gl] if need_x else [gl], go64)
    return (out.detach(),) + (tuple(grads) if need_x else (None,) + tuple(grads))


# ------------------------------------------------------------------------------------------------ (c) sampler backward
WARP_CASES = [
    # source, (Ho, Wo), padding, min_level, image dtype, grid dtype
    (128, (128, 128), "border", 0.0, "f32", torch.float32),
    (256, (96, 160), "reflection", 0.0, "f32", torch.float32),
    (450, (37, 45), "zeros", 1.5, "f32", torch.float32),
    (512, (128, 128), "reflection", 0.0, "f32", torch.float32),     # 512^2: the pyramid is built one level at a time
    (256, (1, 64), "border", 1.5, "f32", torch.float32),
    (256, (64, 1), "zeros", 0.0, "f32", torch.float32),
    (256, (96, 160), "border", 0.0, "bf16", torch.float32),
    (450, (128, 128), "reflection", 1.5, "f16", torch.float32),
    (128, (37, 45), "reflection", 0.0, "bf16", torch.float64),
    (512, (37, 45), "zeros", 1.5, "f16", torch.float32),
]


@pytest.mark.parametrize("size,out_hw,mode,min_level,dt,grid_dt", WARP_CASES,
                         ids=["%d-%dx%d-%s-min%g-%s%s" % (c[0], c[1][0], c[1][1], c[2], c[3], c[4], "-grid64" if c[5] == torch.float64 else "")
                              for c in WARP_CASES])
def test_warp_backward_vs_float64(size, out_hw, mode, min_level, dt, grid_dt):
    """MipmapWarp and Warp backward: grad_grid on decided pixels, grad_x everywhere, against the float64 oracle.  The
    three samples zoom in (level clamped at 0), sit between levels, and zoom out past the last level (clamped)."""
    smp = _smp()
    dtype = DTYPES[dt]
    ho, wo = out_hw
    g = torch.Generator().manual_seed(size * 7 + ho * 3 + wo)
    n = 3
    x = torch.randn(n, 3, size, size, generator=g).to(dtype)
    go = torch.randn(n, 3, ho, wo, generator=g).to(dtype)
    grid = _perturbed_grid(n, size, size, ho, wo, g).to(grid_dt)
    grid64 = grid.float().double()          # what the kernel samples with (it takes the grid in fp32)
    x64, go64 = x.double(), go.double()
    for mip in (True, False):
        xl = x.to(DEV).requires_grad_(True)
        gl = grid.to(DEV).requires_grad_(True)
        if mip:
            out, levels = smp.mipmap_warp(xl, gl, LEVELS, min_level, mode)
        else:
            out = smp.grid_sample_bilinear(xl, gl, mode)
        gx, gg = torch.autograd.grad(out, [xl, gl], go.to(DEV))
        assert gg.dtype == grid_dt and gx.dtype == dtype
        _, gx_o, gg_o = _oracle_warp(x64, grid64, go64, mip, min_level if mip else 0.0, mode)
        ok = S.decided_pixels(grid64, size, size, mode, LEVELS if mip else None, min_level if mip else 0.0)
        frac = ok.double().mean().item()
        if mip:
            lv = S.mipmap_levels(grid64, size, size, LEVELS, min_level)
            assert (lv == max(min_level, 0.0)).any() and (lv == LEVELS - 1).any() and ((lv > min_level) & (lv < LEVELS - 1)).any()
        gg, gx = gg.double().cpu(), gx.double().cpu()
        scale = gg_o[ok].abs().max().item()
        e_grid = (gg - gg_o)[ok[..., None].expand_as(gg)].abs().max().item() / scale
        # grad_x is continuous in the grid: everywhere.  A half-precision image gets its gradient back in its type.
        e_x = ((gx - gx_o).abs() - EPS[dtype] * gx_o.abs()).max().item() / gx_o.abs().max().item()
        _report("warp %s mip=%d" % (dt, mip), decided=frac, grad_grid=e_grid, grad_x=e_x)
        assert frac >= MIN_DECIDED
        assert e_grid <= 1e-3, "grad_grid on decided pixels: rel err %.3e" % e_grid
        assert e_x <= 5e-4, "grad_x: rel err %.3e" % e_x


# ------------------------------------------------------------------------------------------------ flow inputs
FLOW_SHAPES = [(16, 16, 8), (5, 7, 4), (3, 3, 1)]


def _flow_inputs(n, lh, lw, s, gen, with_base, with_alpha):
    low = 0.03 * torch.randn(n, lh, lw, 2, generator=gen)
    mask = torch.randn(n, 9 * s * s, lh, lw, generator=gen)
    base = (torch.eye(2, 3)[None] * (0.6 + 0.8 * torch.rand(n, 1, 1, generator=gen)) + 0.1 * torch.randn(n, 2, 3, generator=gen)) \
        if with_base else None
    alpha = (0.3 + 0.7 * torch.rand(n, generator=gen)) if with_alpha else None
    ident = FL.identity_flow_ref(s * lh, s * lw)
    return low, mask, base, alpha, ident


def _dev(t):
    return None if t is None else t.to(DEV)


def _f64(t):
    return None if t is None else t.double()


# ------------------------------------------------------------------------------------------------ (d) fused = pieces
@pytest.mark.parametrize("lh,lw,s", FLOW_SHAPES)
@pytest.mark.parametrize("with_base", [True, False])
@pytest.mark.parametrize("with_alpha", [True, False])
def test_fused_flow_backward_is_its_pieces_bitwise(lh, lw, s, with_base, with_alpha):
    """stn_sample_flow's backward with the image, the returned grid and the returned delta all in the loss (the TV
    regulariser's path) equals mipmap_warp's backward on the returned grid, followed by flow_compose's backward fed
    that gradient plus the grid's own as g_flow, and g_delta: the same kernels on the same bits, so torch.equal."""
    smp, stn = _smp(), _stn()
    g = torch.Generator().manual_seed(100 * lh + 10 * s + 2 * with_base + with_alpha)
    n, size = 3, 96
    low, mask, base, alpha, ident = [_dev(t) for t in _flow_inputs(n, lh, lw, s, g, with_base, with_alpha)]
    img = (torch.rand(n, 3, size, size, generator=g) * 2 - 1).to(DEV)
    ho, wo = s * lh, s * lw
    go, gf, gd = [torch.randn(n, *shp, generator=g).to(DEV) for shp in ((3, ho, wo), (ho, wo, 2), (ho, wo, 2))]
    for mode in S.PAD_MODES:
        leaves = [t.clone().requires_grad_(True) for t in (low, mask)] + ([base.clone().requires_grad_(True)] if with_base else [])
        out, grid, delta, _ = smp.stn_sample_flow(img, leaves[0], leaves[1], ident, leaves[2] if with_base else None, alpha, s,
                                                  LEVELS, 0.0, mode)
        fused = torch.autograd.grad([out, grid, delta], leaves, [go, gf, gd])
        gl = grid.detach().clone().requires_grad_(True)
        (g_grid,) = torch.autograd.grad(smp.mipmap_warp(img, gl, LEVELS, 0.0, mode)[0], gl, go)
        leaves2 = [t.clone().requires_grad_(True) for t in (low, mask)] + ([base.clone().requires_grad_(True)] if with_base else [])
        d2, f2 = stn.flow_compose(leaves2[0], leaves2[1], ident, leaves2[2] if with_base else None, alpha, s)
        pieces = torch.autograd.grad([d2, f2], leaves2, [gd, g_grid + gf])
        for a, b, name in zip(fused, pieces, ("g_low", "g_mask", "g_base")):
            assert torch.equal(a, b), "%s %s differs from its pieces by %.3e" % (mode, name, (a - b).abs().max().item())
            assert a.abs().max() > 0


@pytest.mark.parametrize("size,out_hw,mode,min_level", [(256, (128, 128), "reflection", 0.0), (450, (37, 45), "border", 1.5),
                                                        (128, (1, 64), "zeros", 0.0), (128, (64, 1), "border", 0.0)])
def test_fused_affine_backward_is_its_pieces(size, out_hw, mode, min_level):
    """stn_sample_affine's d theta (image and returned grid both in the loss) equals F.affine_grid's backward applied to
    mipmap_warp's grid gradient on the returned grid plus the grid's own gradient.  F.affine_grid sums in another order:
    the error is judged against sum_p |grad_grid_p| |basis_p|, the bound of an fp32 sum of those terms."""
    smp = _smp()
    g = torch.Generator().manual_seed(size + out_hw[0])
    n = 4
    ho, wo = out_hw
    theta = _random_thetas(n, size, size, ho, wo, g, spacings=[0.7, 1.8, 3.1, 7.0]).float().to(DEV)
    img = (torch.rand(n, 3, size, size, generator=g) * 2 - 1).to(DEV)
    go, gf = torch.randn(n, 3, ho, wo, generator=g).to(DEV), torch.randn(n, ho, wo, 2, generator=g).to(DEV)
    tl = theta.clone().requires_grad_(True)
    out, grid, _ = smp.stn_sample_affine(img, tl, (ho, wo), LEVELS, min_level, mode)
    (fused,) = torch.autograd.grad([out, grid], [tl], [go, gf])
    gl = grid.detach().clone().requires_grad_(True)
    (g_grid,) = torch.autograd.grad(smp.mipmap_warp(img, gl, LEVELS, min_level, mode)[0], gl, go)
    total = g_grid + gf
    t2 = theta.clone().requires_grad_(True)
    (pieces,) = torch.autograd.grad(F.affine_grid(t2, (n, 3, ho, wo), align_corners=False), t2, total)
    basis = torch.stack([(2 * torch.arange(wo, device=DEV) + 1.0)[None, :].expand(ho, wo) / wo - 1,
                         (2 * torch.arange(ho, device=DEV) + 1.0)[:, None].expand(ho, wo) / ho - 1,
                         torch.ones(ho, wo, device=DEV)], dim=2)
    bound = torch.einsum("nyxi,yxk->nik", total.abs().double(), basis.abs().double())
    # (a single row or column has a zero basis column: both sides must then be exactly zero)
    err = ((fused.double() - pieces.double()).abs() / bound.clamp(min=1e-300)).max().item()
    _report("affine pieces %d %dx%d" % (size, ho, wo), rel_to_abs_sum=err)
    assert err <= 1e-6


# ------------------------------------------------------------------------------------------------ (e) fused forward
AFFINE_FWD = [(256, (128, 128), "border", 0.0, "f32"), (450, (37, 45), "reflection", 1.5, "bf16"),
              (128, (1, 64), "zeros", 0.0, "f32"), (512, (64, 1), "border", 0.0, "f16"), (256, (96, 160), "zeros", 0.0, "f32")]


def _check_forward(what, out, grid, levels, x64, grid_o, mode, min_level, dtype, size, delta=None, delta_o=None):
    out_o, aux = S.mipmap_warp_ref(x64, grid_o, LEVELS, min_level, mode, return_aux=True)
    e_grid = (grid.double().cpu() - grid_o).abs().max().item()
    e_lv = (levels.double().cpu() - aux["levels"]).abs().max().item()
    o = out.double().cpu()
    e_out = ((o - out_o).abs() - EPS[dtype] * out_o.abs()).max().item() / out_o.abs().max().item()
    vals = dict(grid=e_grid, levels=e_lv, out=e_out)
    if delta is not None:
        vals["delta"] = (delta.double().cpu() - delta_o).abs().max().item()
    _report(what, **vals)
    assert e_grid <= 1e-5 and e_lv <= 5e-4 and e_out <= 5e-4
    if delta is not None:
        assert vals["delta"] <= 1e-5


@pytest.mark.parametrize("size,out_hw,mode,min_level,dt", AFFINE_FWD)
def test_fused_affine_forward_vs_float64(size, out_hw, mode, min_level, dt):
    """stn_sample_affine's grid, levels and output against affine_grid_ref -> mipmap_warp_ref in float64, with seeded
    random thetas, at outputs that are not a multiple of the 32x8 tile (its one-pixel halo ring)."""
    smp = _smp()
    dtype = DTYPES[dt]
    ho, wo = out_hw
    g = torch.Generator().manual_seed(size * 5 + ho + wo)
    n = 3
    theta = _random_thetas(n, size, size, ho, wo, g).float()
    x = (torch.rand(n, 3, size, size, generator=g) * 2 - 1).to(dtype)
    out, grid, levels = smp.stn_sample_affine(x.to(DEV), theta.to(DEV), (ho, wo), LEVELS, min_level, mode)
    grid_o = S.affine_grid_ref(theta.double(), (n, 3, ho, wo))
    _check_forward("affine fwd %d %dx%d %s" % (size, ho, wo, dt), out, grid, levels, x.double(), grid_o, mode, min_level,
                   dtype, size)


FLOW_FWD = [(256, (16, 16, 8), "reflection", True, False, "f32"), (96, (5, 7, 4), "border", True, True, "bf16"),
            (64, (3, 3, 1), "zeros", False, True, "f32"), (450, (5, 7, 4), "reflection", False, False, "f32")]


@pytest.mark.parametrize("size,flow_shape,mode,with_base,with_alpha,dt", FLOW_FWD)
def test_fused_flow_forward_vs_float64(size, flow_shape, mode, with_base, with_alpha, dt):
    """stn_sample_flow's grid, delta, levels and output against flow_compose_ref -> mipmap_warp_ref in float64."""
    smp = _smp()
    dtype = DTYPES[dt]
    lh, lw, s = flow_shape
    g = torch.Generator().manual_seed(size + lh * 10 + s)
    n = 3
    low, mask, base, alpha, ident = _flow_inputs(n, lh, lw, s, g, with_base, with_alpha)
    x = (torch.rand(n, 3, size, size, generator=g) * 2 - 1).to(dtype)
    out, grid, delta, levels = smp.stn_sample_flow(x.to(DEV), low.to(DEV), mask.to(DEV), ident.to(DEV), _dev(base), _dev(alpha), s,
                                                   LEVELS, 0.0, mode)
    delta_o, grid_o = FL.flow_compose_ref(low.double(), mask.double(), ident.double(), _f64(base), _f64(alpha), s)
    _check_forward("flow fwd %d %dx%dx%d %s" % (size, lh, lw, s, dt), out, grid, levels, x.double(), grid_o, mode, 0.0,
                   dtype, size, delta, delta_o)


# ------------------------------------------------------------------------------------------------ bounds for reductions
def _flow_abs_adjoint(low, mask, ident, base, alpha, s, a, b):
    """Sums of the absolute per-pixel contributions to (g_low, g_mask, g_base) of flow composition's backward, for
    non-negative gradients `a` at the flow (grid) and `b` at delta, each (N, sH, sW, 2): every product of the chain
    rule with its factors replaced by their absolute values.  float64."""
    n, h, w, _ = low.shape
    if alpha is not None:
        a = a * alpha.abs().reshape(n, 1, 1, 1)
    delta = FL.upsample_flow_ref(low, mask, s)
    b_base = None
    if base is not None:
        f = ident + delta
        fk = torch.cat([f.abs(), torch.ones_like(f[..., :1])], dim=-1)
        b_base = torch.einsum("nyxi,nyxk->nik", a, fk)
        a = torch.einsum("nyxi,nij->nyxj", a, base[:, :, :2].abs())
    e = a + b
    lo = low.clone().requires_grad_(True)
    (b_low,) = torch.autograd.grad(FL.upsample_flow_ref(lo, mask, s), lo, e)    # its coefficients s * p_k are >= 0
    p = torch.softmax(mask.reshape(n, 9, s, s, h, w), dim=1)
    padded = F.pad(s * low.abs().permute(0, 3, 1, 2), (1, 1, 1, 1))
    e6 = e.reshape(n, h, s, w, s, 2).permute(0, 5, 2, 4, 1, 3)                   # (N, 2, sy, sx, H, W)
    t = torch.stack([(e6 * padded[:, :, None, None, k // 3:k // 3 + h, k % 3:k % 3 + w]).sum(dim=1) for k in range(9)], dim=1)
    b_mask = p * (t + (p * t).sum(dim=1, keepdim=True))                          # |p_k (t_k - sum_j p_j t_j)|
    return b_low, b_mask.reshape(mask.shape), b_base


def _check_reduction(what, got, want, bound, allowance, tol):
    """|got - want| <= tol * bound + allowance, elementwise."""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    diff = (got - want).abs()
    bound = bound.clamp(min=1e-300)
    err = ((diff - allowance) / bound).max().item()
    _report(what, err_over_abs_sum=err, raw_err_over_abs_sum=(diff / bound).max().item(),
            allowance_over_abs_sum=(allowance / bound).max().item())
    assert err <= tol, "%s: error %.3e of the sum of absolute contributions" % (what, err)


# ------------------------------------------------------------------------------------------------ (f) head gradients
HEAD_CASES = [
    # batch, source, affine output, flow (lh, lw, s), padding, min_level, alpha
    (32, 256, (128, 128), (16, 16, 8), "reflection", 0.0, False),    # the benchmark's shapes
    (3, 450, (37, 45), (5, 7, 4), "zeros", 1.5, True),
    (2, 128, (64, 1), (3, 3, 1), "border", 0.0, True),
]


@pytest.mark.parametrize("n,size,out_hw,flow_shape,mode,min_level,with_alpha", HEAD_CASES)
def test_head_parameter_gradients_vs_float64(n, size, out_hw, flow_shape, mode, min_level, with_alpha):
    """g_theta (similarity head), g_low, g_mask and g_base (flow head) end to end against float64 autograd of the oracle
    composition.  Error is measured against the sum of the absolute per-pixel contributions (not the result's own
    maximum: these are sums of many terms of random sign), with an allowance for what the undecided pixels could
    contribute: their |grid gradient| from the oracle plus the kernel's."""
    smp = _smp()
    g = torch.Generator().manual_seed(n * 1000 + size)
    img = torch.rand(n, 3, size, size, generator=g) * 2 - 1
    x64 = img.double()
    # similarity head: stn_sample_affine
    ho, wo = out_hw
    theta = _random_thetas(n, size, size, ho, wo, g, spacings=[(0.8, 1.7, 2.9, 4.6)[i % 4] for i in range(n)]).float()
    go = torch.randn(n, 3, ho, wo, generator=g)
    tl = theta.to(DEV).requires_grad_(True)
    out, grid, _ = smp.stn_sample_affine(img.to(DEV), tl, (ho, wo), LEVELS, min_level, mode)
    (g_theta,) = torch.autograd.grad(out, tl, go.to(DEV))
    gl = grid.detach().clone().requires_grad_(True)
    (gg_k,) = torch.autograd.grad(smp.mipmap_warp(img.to(DEV), gl, LEVELS, min_level, mode)[0], gl, go.to(DEV))
    t64 = theta.double().requires_grad_(True)
    grid_o = S.affine_grid_ref(t64, (n, 3, ho, wo))
    out_o = S.mipmap_warp_ref(x64, grid_o, LEVELS, min_level, mode)
    g_theta_o, gg_o = torch.autograd.grad(out_o, [t64, grid_o], go.double())
    ok = S.decided_pixels(grid_o.detach(), size, size, mode, LEVELS, min_level, axis_ties=True)
    basis = torch.stack([(2 * torch.arange(wo, dtype=torch.float64) + 1)[None, :].expand(ho, wo) / wo - 1,
                         (2 * torch.arange(ho, dtype=torch.float64) + 1)[:, None].expand(ho, wo) / ho - 1,
                         torch.ones(ho, wo, dtype=torch.float64)], dim=2).abs()
    bound = torch.einsum("nyxi,yxk->nik", gg_o.abs(), basis)
    undecided = (~ok)[..., None] * (gg_o.abs() + gg_k.double().cpu().abs())
    allowance = torch.einsum("nyxi,yxk->nik", undecided, basis)
    frac = ok.double().mean().item()
    _report("head affine n=%d %d" % (n, size), decided=frac)
    assert frac >= MIN_DECIDED
    _check_reduction("g_theta", g_theta, g_theta_o, bound, allowance, 1e-4)

    # flow head: stn_sample_flow with the image and delta (the TV term) in the loss
    lh, lw, s = flow_shape
    low, mask, base, alpha, ident = _flow_inputs(n, lh, lw, s, g, True, with_alpha)
    fo, fw = s * lh, s * lw
    go, gd = torch.randn(n, 3, fo, fw, generator=g), torch.randn(n, fo, fw, 2, generator=g)
    leaves = [t.to(DEV).requires_grad_(True) for t in (low, mask, base)]
    out, grid, delta, _ = smp.stn_sample_flow(img.to(DEV), leaves[0], leaves[1], ident.to(DEV), leaves[2], _dev(alpha), s,
                                              LEVELS, min_level, mode)
    got = torch.autograd.grad([out, delta], leaves, [go.to(DEV), gd.to(DEV)])
    gl = grid.detach().clone().requires_grad_(True)
    (gg_k,) = torch.autograd.grad(smp.mipmap_warp(img.to(DEV), gl, LEVELS, min_level, mode)[0], gl, go.to(DEV))
    leaves_o = [t.double().requires_grad_(True) for t in (low, mask, base)]
    delta_o, grid_o = FL.flow_compose_ref(leaves_o[0], leaves_o[1], ident.double(), leaves_o[2], _f64(alpha), s)
    out_o = S.mipmap_warp_ref(x64, grid_o, LEVELS, min_level, mode)
    want = torch.autograd.grad([out_o, delta_o], leaves_o + [grid_o], [go.double(), gd.double()])
    gg_o = want[3]
    ok = S.decided_pixels(grid_o.detach(), size, size, mode, LEVELS, min_level)
    frac = ok.double().mean().item()
    _report("head flow n=%d %d" % (n, size), decided=frac)
    assert frac >= MIN_DECIDED
    consts = (low.double(), mask.double(), ident.double(), base.double(), _f64(alpha), s)
    bounds = _flow_abs_adjoint(*consts, gg_o.abs(), gd.double().abs())
    allow = list(_flow_abs_adjoint(*consts, (~ok)[..., None] * (gg_o.abs() + gg_k.double().cpu().abs()), torch.zeros_like(gg_o)))
    # An element of g_mask is one pixel's term, not a sum over pixels: its error is that of the pixel's grid gradient, a
    # sum over channels, corners and levels that may cancel.  It is judged against the largest bound of its sample.
    bounds = list(bounds)
    bounds[1] = bounds[1].flatten(1).max(dim=1).values.reshape(n, 1, 1, 1).expand_as(bounds[1])
    for name, a, w_, bd, al, tol in zip(("g_low", "g_mask", "g_base"), got, want[:3], bounds, allow, (1e-4, 2e-4, 1e-4)):
        _check_reduction(name, a, w_, bd, al, tol)


# ------------------------------------------------------------------------------------------------ (g) flow backward alone
FLOW_BWD = [
    # N, H, W, S, base, alpha   (per-sample terms S*S*H*W vs the 256-thread reduction block)
    (1, 1, 1, 2, True, True),        # 4 terms; every tap but the centre lies outside the grid
    (33, 1, 5, 8, True, False),      # 320
    (1, 4, 1, 1, False, True),       # 4
    (33, 3, 5, 1, True, True),       # 15
    (1, 4, 5, 8, True, True),        # 1280
    (33, 16, 16, 2, True, False),    # 1024
    (2, 16, 16, 8, False, False),
]


@pytest.mark.parametrize("n,h,w,s,with_base,with_alpha", FLOW_BWD)
def test_flow_compose_backward_vs_float64(n, h, w, s, with_base, with_alpha):
    """flow_compose's backward (g_low, g_mask, g_base) against float64 autograd of flow_compose_ref, with g_delta and
    g_flow both live.  The operation is smooth: every element is within a small multiple of fp32 rounding of the
    sum of its absolute contributions."""
    stn = _stn()
    g = torch.Generator().manual_seed(n * 100 + h * 10 + w + s)
    low, mask, base, alpha, ident = _flow_inputs(n, h, w, s, g, with_base, with_alpha)
    low = low * 30           # flows of a few pixels: the taps' values matter as much as the weights
    gd, gf = torch.randn(n, s * h, s * w, 2, generator=g), torch.randn(n, s * h, s * w, 2, generator=g)
    leaves = [t.to(DEV).requires_grad_(True) for t in (low, mask)] + ([base.to(DEV).requires_grad_(True)] if with_base else [])
    d, f = stn.flow_compose(leaves[0], leaves[1], ident.to(DEV), leaves[2] if with_base else None, _dev(alpha), s)
    got = torch.autograd.grad([d, f], leaves, [gd.to(DEV), gf.to(DEV)])
    leaves_o = [t.double().requires_grad_(True) for t in (low, mask)] + ([base.double().requires_grad_(True)] if with_base else [])
    d_o, f_o = FL.flow_compose_ref(leaves_o[0], leaves_o[1], ident.double(), leaves_o[2] if with_base else None, _f64(alpha), s)
    assert (d.double().cpu() - d_o).abs().max() <= 1e-5 * d_o.abs().max() and (f.double().cpu() - f_o).abs().max() <= 1e-5 * f_o.abs().max()
    want = torch.autograd.grad([d_o, f_o], leaves_o, [gd.double(), gf.double()])
    bounds = _flow_abs_adjoint(low.double(), mask.double(), ident.double(), _f64(base), _f64(alpha), s, gf.double().abs(),
                               gd.double().abs())
    zero = torch.zeros(())
    for name, a, w_, bd in zip(("g_low", "g_mask", "g_base"), got, want, bounds):
        _check_reduction("flow bwd %s" % name, a, w_, bd, zero, 1e-5)


# ------------------------------------------------------------------------------------------------ (h) empty inputs
def _poison(*shapes):
    """Fill the caching allocator's free blocks of these shapes (fp32) with NaN, so that an output allocated with
    torch.empty and then not written shows up as NaN rather than as whatever the block held."""
    held = [torch.full(shp, float("nan"), device=DEV) for shp in shapes for _ in range(4)]
    del held


def test_zero_channels_write_every_output():
    """With C == 0 the grid, the flow, the levels and the grid gradient are still defined: they do not depend on the
    channels.  Warp's and MipmapWarp's grid gradient is zero, as from F.grid_sample; the fused forward's grid, delta and
    levels equal those of a C = 3 call.  (Outputs are allocated with torch.empty: the kernels must write them.)"""
    smp = _smp()
    g = torch.Generator().manual_seed(9)
    n, size, ho, wo = 2, 64, 24, 40
    grid = _perturbed_grid(n, size, size, ho, wo, g).to(DEV)
    x0 = torch.zeros(n, 0, size, size, device=DEV)
    x3 = torch.rand(n, 3, size, size, generator=g).to(DEV)
    for mip in (False, True):
        for mode in S.PAD_MODES:
            _poison((n, ho, wo, 2), (n, ho, wo))
            gl = grid.clone().requires_grad_(True)
            if mip:
                out, levels = smp.mipmap_warp(x0, gl, LEVELS, 0.0, mode)
                _, levels3 = smp.mipmap_warp(x3, grid, LEVELS, 0.0, mode)
                assert torch.equal(levels, levels3), "levels with C = 0"
            else:
                out = smp.grid_sample_bilinear(x0, gl, mode)
            assert out.shape == (n, 0, ho, wo)
            _poison((n, ho, wo, 2))
            (gg,) = torch.autograd.grad(out, gl, torch.zeros_like(out))
            assert torch.equal(gg, torch.zeros_like(gg)), "grad_grid with C = 0 (mip %d, %s): %s" % (mip, mode, gg.flatten()[:4])
    cg = grid.detach().cpu().requires_grad_(True)
    (gref,) = torch.autograd.grad(F.grid_sample(torch.zeros(n, 0, size, size), cg, align_corners=False), cg,
                                  torch.zeros(n, 0, ho, wo))
    assert torch.equal(gref, torch.zeros_like(gref))
    # the fused forward: affine and flow
    theta = _random_thetas(n, size, size, ho, wo, g).float().to(DEV)
    _poison((n, ho, wo, 2), (n, ho, wo))
    out0, grid0, lv0 = smp.stn_sample_affine(x0, theta, (ho, wo), LEVELS, 0.0, "border")
    _, grid3, lv3 = smp.stn_sample_affine(x3, theta, (ho, wo), LEVELS, 0.0, "border")
    assert out0.shape == (n, 0, ho, wo) and torch.equal(grid0, grid3) and torch.equal(lv0, lv3)
    low, mask, base, alpha, ident = [_dev(t) for t in _flow_inputs(n, 5, 7, 4, g, True, True)]
    _poison((n, 20, 28, 2), (n, 20, 28))
    out0, grid0, delta0, lv0 = smp.stn_sample_flow(x0, low, mask, ident, base, alpha, 4, LEVELS, 0.0, "reflection")
    _, grid3, delta3, lv3 = smp.stn_sample_flow(x3, low, mask, ident, base, alpha, 4, LEVELS, 0.0, "reflection")
    assert torch.equal(grid0, grid3) and torch.equal(delta0, delta3) and torch.equal(lv0, lv3)
    # the fused backward: only the returned grid carries a gradient to theta
    tl = theta.clone().requires_grad_(True)
    out0, grid0, _ = smp.stn_sample_affine(x0, tl, (ho, wo), LEVELS, 0.0, "border")
    gf = torch.randn(n, ho, wo, 2, generator=g).to(DEV)
    (gt,) = torch.autograd.grad([out0, grid0], [tl], [torch.zeros_like(out0), gf])
    t2 = theta.clone().requires_grad_(True)
    (gt_ref,) = torch.autograd.grad(F.affine_grid(t2, (n, 3, ho, wo), align_corners=False), t2, gf)
    assert torch.allclose(gt, gt_ref, rtol=1e-5, atol=1e-5 * gt_ref.abs().max().item())


def test_zero_batch():
    """N == 0: every entry point returns empty tensors of the right shapes (nothing to write)."""
    smp, stn = _smp(), _stn()
    x = torch.zeros(0, 3, 64, 64, device=DEV)
    grid = torch.zeros(0, 24, 40, 2, device=DEV, requires_grad=True)
    out, levels = smp.mipmap_warp(x, grid, LEVELS, 0.0, "border")
    assert out.shape == (0, 3, 24, 40) and levels.shape == (0, 24, 40)
    (gg,) = torch.autograd.grad(out, grid, torch.zeros_like(out))
    assert gg.shape == grid.shape
    theta = torch.zeros(0, 2, 3, device=DEV, requires_grad=True)
    out, grid2, levels = smp.stn_sample_affine(x, theta, (24, 40), LEVELS, 0.0, "border")
    assert out.shape == (0, 3, 24, 40) and grid2.shape == (0, 24, 40, 2) and levels.shape == (0, 24, 40)
    (gt,) = torch.autograd.grad([out, grid2], [theta], [torch.zeros_like(out), torch.zeros_like(grid2)])
    assert gt.shape == theta.shape
    low = torch.zeros(0, 5, 7, 2, device=DEV, requires_grad=True)
    mask = torch.zeros(0, 144, 5, 7, device=DEV, requires_grad=True)
    ident = FL.identity_flow_ref(20, 28).to(DEV)
    out, flow, delta, levels = smp.stn_sample_flow(x, low, mask, ident, None, None, 4, LEVELS, 0.0, "border")
    assert out.shape == (0, 3, 20, 28) and flow.shape == (0, 20, 28, 2) and delta.shape == (0, 20, 28, 2)
    gl, gm = torch.autograd.grad([out, flow, delta], [low, mask], [torch.zeros_like(out), torch.zeros_like(flow), torch.zeros_like(delta)])
    assert gl.shape == low.shape and gm.shape == mask.shape
    d, f = stn.flow_compose(low, mask, ident, None, None, 4)
    assert d.shape == (0, 20, 28, 2) and f.shape == (0, 20, 28, 2)
