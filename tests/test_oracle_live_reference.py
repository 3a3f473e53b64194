"""CPU: seeded random SWEEPS of the oracle restatement against the reference itself (its native CPU branches).  The fixtures
of oracle/make_golden.py pin a fixed list of cases; these sweeps widen the pin -- hundreds of parameter tuples per op (sizes,
strides, pads incl. negative, filter shapes, padding modes, head counts).  What the reference computed for each case is kept
in tests/golden/sweep_*.npz (conftest.Pinned; GG_RECORD_GOLDEN=1 with the reference checkout importable recomputes it)."""
import importlib
import random

import torch
import torch.nn.functional as F

from conftest import Pinned
from oracle import flow as FL
from oracle import refimport
from oracle import sampling as S
from oracle import stylegan2_ops as so


def _err(a, b):
    return (a - b).abs().max().item() / max(1.0, b.abs().max().item())


def _ref(module):
    """A module of the reference checkout (only reached while recording)."""
    refimport.import_reference()
    torch.Tensor.cuda = lambda self, *a, **k: self   # reference FlowHead.__init__ calls .cuda() (warping_heads.py:158)
    return importlib.import_module(module)


def test_upfirdn2d_sweep_vs_reference_native_branch():
    """reference upfirdn2d() on CPU tensors takes upfirdn2d_native (upfirdn2d.py:146-149,159-200)."""
    pin = Pinned("sweep_upfirdn2d")
    rng = random.Random(101)
    gen = torch.Generator().manual_seed(101)
    done = 0
    while done < 150:
        n, c = rng.randint(1, 2), rng.randint(1, 3)
        h, w = rng.randint(4, 21), rng.randint(4, 21)
        kh = kw = rng.randint(1, 5)
        if rng.random() < 0.3:
            kw = rng.randint(1, 5)
        up, down = rng.randint(1, 3), rng.randint(1, 3)
        pad = (rng.randint(-2, 4), rng.randint(-2, 4))
        if min(h * up + pad[0] + pad[1] - kh, w * up + pad[0] + pad[1] - kw) < 0:
            continue
        if h * up - max(-pad[0], 0) - max(-pad[1], 0) <= 0 or w * up - max(-pad[0], 0) - max(-pad[1], 0) <= 0:
            continue   # the crop of a negative pad would leave nothing
        x = torch.randn(n, c, h, w, generator=gen)
        k = torch.randn(kh, kw, generator=gen)
        got, want = pin("case%d" % done, so.upfirdn2d_ref(x, k, up=up, down=down, pad=pad),
                        lambda: _ref("models.stylegan2.op.upfirdn2d").upfirdn2d(x, k, up=up, down=down, pad=pad))
        assert _err(got, want) < 1e-5, (x.shape, k.shape, up, down, pad)
        done += 1
    pin.save()


def test_fused_leaky_relu_sweep_vs_reference_native_branch():
    """reference fused_leaky_relu() on CPU (fused_act.py:86-94; the branch hard-codes slope 0.2) for 2-D .. 5-D inputs."""
    pin = Pinned("sweep_fused_leaky_relu")
    rng = random.Random(202)
    gen = torch.Generator().manual_seed(202)
    for i in range(60):
        dims = rng.randint(2, 5)
        shape = [rng.randint(1, 4), rng.randint(1, 9)] + [rng.randint(1, 6) for _ in range(dims - 2)]
        x = torch.randn(*shape, generator=gen)
        b = torch.randn(shape[1], generator=gen)
        scale = rng.choice([1.0, 2 ** 0.5, 0.37])
        go = torch.randn(x.shape, generator=gen)
        out = so.fused_leaky_relu_ref(x, b, 0.2, scale)
        gx, gb = so.fused_leaky_relu_backward_ref(go, out, 0.2, scale)

        def reference():   # and its autograd: grad_input / grad_bias of FusedLeakyReLUFunctionBackward == autograd of the CPU branch
            xr, br = x.clone().requires_grad_(True), b.clone().requires_grad_(True)
            want = _ref("models.stylegan2.op.fused_act").fused_leaky_relu(xr, br, 0.2, scale)
            return (want.detach(),) + torch.autograd.grad(want, [xr, br], go)
        (o, o_ref), (gx, gx_ref), (gb, gb_ref) = pin("case%d" % i, (out, gx, gb), reference)
        assert _err(o, o_ref) < 1e-6, shape
        assert _err(gx, gx_ref) < 1e-6 and _err(gb, gb_ref) < 1e-5, shape
    pin.save()


def _random_grid(gen, rng, n, res):
    """A similarity warp (scale 0.5 .. 3.5: magnification to strong minification) plus a smooth perturbation."""
    ang = torch.rand(n, generator=gen) * 6.283
    sc = 0.5 + 3.0 * torch.rand(n, generator=gen)
    theta = torch.stack([torch.stack([sc * ang.cos(), -sc * ang.sin(), torch.rand(n, generator=gen) - 0.5], 1),
                         torch.stack([sc * ang.sin(), sc * ang.cos(), torch.rand(n, generator=gen) - 0.5], 1)], 1)
    base = F.affine_grid(theta, (n, 1, res, res), align_corners=False)
    coarse = torch.randn(n, 2, 4, 4, generator=gen)
    bump = F.interpolate(coarse, size=(res, res), mode="bicubic", align_corners=False).permute(0, 2, 3, 1)
    return (base + rng.choice([0.0, 0.03, 0.2]) * bump).contiguous()


def test_mipmap_warp_and_warp_sweep_vs_reference_modules():
    """reference MipmapWarp / Warp modules (antialiased_sampling.py:9-238) on CPU: outputs, level maps, autograd."""
    pin = Pinned("sweep_mipmap_warp")
    rng = random.Random(303)
    gen = torch.Generator().manual_seed(303)
    for i in range(40):
        n, c = rng.randint(1, 2), rng.choice([1, 3])
        size = rng.choice([8, 16, 20, 32, 45, 52, 64])
        res = rng.choice([6, 8, 16, 24, 32])
        mode = rng.choice(["border", "reflection", "zeros"])
        levels = rng.choice([3.5, 2.0, 8])
        min_level = rng.choice([0.0, 0.0, 0.5])
        x = torch.randn(n, c, size, size, generator=gen, requires_grad=True)
        grid = _random_grid(gen, rng, n, res).requires_grad_(True)
        xo, go_ = x.detach().clone().requires_grad_(True), grid.detach().clone().requires_grad_(True)
        got, aux = S.mipmap_warp_ref(xo, go_, levels, min_level, mode, return_aux=True)
        case = (i, n, c, size, res, mode, levels, min_level)
        go = torch.randn(got.shape, generator=gen)
        gx, gg = torch.autograd.grad(got, [xo, go_], go)

        def reference():
            A = _ref("models.spatial_transformers.antialiased_sampling")
            want = A.MipmapWarp(levels)(x, grid, min_level=min_level, padding_mode=mode)
            return (want.detach(),) + torch.autograd.grad(want, [x, grid], go) + (A.Warp()(x, grid, padding_mode=mode).detach(),)
        pairs = pin("case%d" % i, (got, gx, gg, S.warp_ref(x.detach(), grid.detach(), mode)), reference)
        (got, want), (gx, gx_ref), (gg, gg_ref), (warped, warped_ref) = pairs
        assert _err(got, want) < 1e-5, case
        assert _err(gx, gx_ref) < 5e-5 and _err(gg, gg_ref) < 5e-4, case
        assert _err(warped, warped_ref) < 1e-5, case
    pin.save()


def test_bilinear_downsample_sweep_vs_reference_module():
    pin = Pinned("sweep_bilinear_downsample")
    gen = torch.Generator().manual_seed(404)
    for stride in (2, 3, 4, 8):
        for size in (stride * 4, stride * 7, stride * 16):
            x = torch.randn(2, 3, size, size, generator=gen)
            got, want = pin("s%d.%d" % (stride, size), S.bilinear_downsample_ref(x, stride),
                            lambda: _ref("models.spatial_transformers.antialiased_sampling").BilinearDownsample(stride, 3)(x))
            assert _err(got, want) < 1e-6, (stride, size)
    pin.save()


def test_flow_composition_sweep_vs_reference_functions():
    """FlowHead.upsample_flow + apply_affine + identity + alpha lerp (warping_heads.py:180-193,240-244,268-277)."""
    pin = Pinned("sweep_flow_composition")
    rng = random.Random(505)
    gen = torch.Generator().manual_seed(505)

    class _Head:   # upsample_flow only reads this attribute (the constructor needs CUDA: warping_heads.py:158)
        flow_downsample = 8

    for i in range(30):
        n, h, w, s = rng.randint(1, 4), rng.randint(2, 9), rng.randint(2, 9), rng.choice([2, 4, 8])
        _Head.flow_downsample = s
        low = 0.1 * torch.randn(n, h, w, 2, generator=gen)
        mask = 2.0 * torch.randn(n, 9 * s * s, h, w, generator=gen)
        base = torch.eye(2, 3)[None] + 0.3 * torch.randn(n, 2, 3, generator=gen)
        alpha = torch.rand(n, generator=gen) if rng.random() < 0.5 else None
        ident = FL.identity_flow_ref(s * h, s * w)

        def reference():
            wh = _ref("models.spatial_transformers.warping_heads")
            delta_ref = wh.FlowHead.upsample_flow(_Head, low, mask)
            flow_ref = wh.apply_affine(base, ident + delta_ref)
            if alpha is not None:
                flow_ref = ident.lerp(flow_ref, alpha[:, None, None, None])
            return delta_ref, flow_ref
        (delta, delta_ref), (flow, flow_ref) = pin("case%d" % i, FL.flow_compose_ref(low, mask, ident, base, alpha, s), reference)
        assert _err(delta, delta_ref) < 1e-6 and _err(flow, flow_ref) < 1e-6, (n, h, w, s, alpha is not None)
    pin.save()


def test_similarity_matrices_and_affine_grid_sweep():
    pin = Pinned("sweep_similarity_matrices")
    gen = torch.Generator().manual_seed(606)
    for heads in (1, 2, 4):
        params = 1.5 * torch.randn(7, 4 * heads, generator=gen)
        got, want = pin("heads%d" % heads, FL.similarity_matrix_ref(params), lambda: _ref(
            "models.spatial_transformers.warping_heads").SimilarityHead.make_affine_matrix(*torch.split(params, heads, dim=1)))
        assert _err(got, want) < 1e-6, heads
    pin.save()
    for res in ((5, 7), (16, 16), (33, 12)):
        theta = torch.randn(3, 2, 3, generator=gen)
        assert _err(S.affine_grid_ref(theta, (3, 1) + res), F.affine_grid(theta, (3, 1) + res, align_corners=False)) < 1e-6, res


def test_generator_mirror_sweep_vs_reference_module():
    """This repo's Generator (host code of the product) on the oracle op set vs the reference Generator, same seeded weights,
    latents and noise, over sizes / widths / mapping depths; also the w-space entry and truncation."""
    from gangealing_b200.stylegan2 import Generator
    from oracle import opset
    cpu = opset.cpu_ops()
    pin = Pinned("sweep_generator")
    gen = torch.Generator().manual_seed(707)
    for size, dim, n_mlp, mult in ((8, 16, 1, 2), (16, 32, 2, 1), (32, 24, 3, 2), (64, 32, 2, 1)):
        m = opset.fill_parameters(Generator(size, dim, n_mlp, channel_multiplier=mult, ops=cpu).eval(), size)
        z = torch.randn(2, dim, generator=gen)
        noise = [torch.randn(2, 1, n.shape[2], n.shape[3], generator=gen) for n in m.make_noise(1)]
        with torch.no_grad():
            img_m, lat_m = m([z], noise=noise, return_latents=True)
            mean = lat_m.mean(dim=(0, 1))[None]
            b_trunc, _ = m([z], noise=noise, truncation=0.6, truncation_latent=mean, inject_index=2)
            b_w, _ = m([lat_m], input_is_latent=True, noise=noise)

            def reference():
                r = opset.fill_parameters(_ref("models.stylegan2.networks").Generator(size, dim, n_mlp, channel_multiplier=mult).eval(), size)
                img_r, lat_r = r([z], noise=noise, return_latents=True)
                a_trunc, _ = r([z], noise=noise, truncation=0.6, truncation_latent=mean, inject_index=2)
                a_w, _ = r([lat_m], input_is_latent=True, noise=noise)
                return lat_r, img_r, a_trunc, a_w
            (lat_m, lat_r), (img_m, img_r), (b, a), (bw, aw) = pin("g%d" % size, (lat_m, img_m, b_trunc, b_w), reference)
            assert _err(lat_m, lat_r) < 1e-6 and _err(img_m, img_r) < 1e-5, (size, dim, n_mlp, mult)
            assert _err(b, a) < 1e-5, ("truncation", size)
            assert _err(bw, aw) < 1e-5, ("w entry", size)
    pin.save()


def test_stn_mirror_sweep_vs_reference_module():
    """This repo's get_stn(...) on the oracle op set vs the reference's, same seeded weights: transforms, head counts,
    supersize, padding modes, output resolution, similarity iterations."""
    from gangealing_b200.stn import get_stn
    from oracle import opset
    cpu = opset.cpu_ops()
    pin = Pinned("sweep_stn")
    gen = torch.Generator().manual_seed(808)
    cases = [
        (["similarity"], 32, 32, 1, "border", {}),
        (["similarity"], 32, 64, 1, "reflection", {"iters": 2}),     # (the reference cannot iterate a multi-head STN)
        (["similarity"], 32, 64, 2, "reflection", {}),
        (["similarity"], 64, 64, 1, "zeros", {"output_resolution": 48}),
        (["similarity", "flow"], 64, 64, 1, "border", {}),
        (["similarity", "flow"], 64, 128, 2, "reflection", {}),
        (["similarity", "flow"], 64, 64, 3, "border", {"output_resolution": 96}),
        (["flow"], 64, 64, 1, "border", {}),
    ]
    for i, (transforms, flow_size, supersize, heads, mode, kw) in enumerate(cases):
        args = dict(flow_size=flow_size, supersize=supersize, channel_multiplier=0.25, num_heads=heads)
        m = opset.fill_parameters(get_stn(list(transforms), ops=cpu, **args).eval(), 900 + i, gain=0.3)
        x = torch.randn(2, 3, supersize, supersize, generator=gen)

        def reference():
            get_ref = _ref("models.spatial_transformers.spatial_transformer").get_stn
            r = opset.fill_parameters(get_ref(list(transforms), **args).eval(), 900 + i, gain=0.3)
            with torch.no_grad():
                return r(x, return_warp=True, return_flow=True, padding_mode=mode, **kw)
        with torch.no_grad():
            got = m(x, return_warp=True, return_flow=True, padding_mode=mode, **kw)
        assert len(got) == 3
        for j, (a, b) in enumerate(pin("case%d" % i, got, reference)):
            assert _err(a, b) < 2e-4, (transforms, flow_size, supersize, heads, mode, kw, j)
    pin.save()
