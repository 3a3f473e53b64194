"""Warp / MipmapWarp / BilinearDownsample -- drop-ins for reference
models/spatial_transformers/antialiased_sampling.py on sm_100a.

`MipmapWarp(max_num_levels).forward(inputs, grid, min_level=0.0, padding_mode='border')` and
`Warp().forward(inputs, grid, padding_mode='border')` keep the reference call signatures, the
`blur_filter` buffer and the `levels_map` attribute.  One fused kernel per direction
(gg_mipmap_warp_forward / _backward) replaces the ~30 launches and the `.item()` host sync of the
reference's forward (antialiased_sampling.py:35-60); see csrc/warp.cu for the algorithm.
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import _lib


def feasible_levels(h, w, wanted):
    """How many pyramid levels (beyond level 0) a source of this size can host (<= wanted)."""
    lib = _lib.load()
    e = wanted
    while e > 0 and lib.gg_mipmap_pyramid_elems(1, h, w, e) < 0:
        e -= 1
    return e


class _MipmapWarp(Function):
    @staticmethod
    def forward(ctx, inputs, grid, max_level, min_level, pad_mode, extra):
        _lib.require_cuda(inputs, grid)
        if inputs.dim() != 4 or grid.dim() != 4 or grid.shape[-1] != 2 or grid.shape[0] != inputs.shape[0]:
            raise RuntimeError("warp: expected inputs (N, C, H, W) and grid (N, Ho, Wo, 2), got %s and %s" %
                               (tuple(inputs.shape), tuple(grid.shape)))
        lib = _lib.load()
        x = inputs.contiguous()
        g = grid.float().contiguous()
        n, c, hs, ws = x.shape
        ho, wo = g.shape[1], g.shape[2]
        code = _lib.dtype_code(x)
        st = _lib.stream()
        pyr = None
        if extra > 0:
            elems = lib.gg_mipmap_pyramid_elems(n * c, hs, ws, extra)
            if elems < 0:
                raise RuntimeError("MipmapWarp: a %dx%d source cannot host %d mip levels" % (hs, ws, extra))
            pyr = torch.empty(max(int(elems), 1), dtype=torch.float32, device=x.device)
            _lib.check(lib.gg_mipmap_build(pyr.data_ptr(), x.data_ptr(), code, n * c, hs, ws, extra, st), "gg_mipmap_build")
        out = torch.empty((n, c, ho, wo), dtype=x.dtype, device=x.device)
        levels = torch.empty((n, ho, wo), dtype=torch.float32, device=x.device) if extra > 0 else None
        rc = lib.gg_mipmap_warp_forward(out.data_ptr(), _lib.ptr(levels), x.data_ptr(), _lib.ptr(pyr), g.data_ptr(), code,
                                        n, c, hs, ws, ho, wo, extra, max_level, min_level, pad_mode, st)
        _lib.check(rc, "gg_mipmap_warp_forward")
        ctx.save_for_backward(x, g, pyr)
        ctx.cfg = (max_level, min_level, pad_mode, extra, grid.dtype)
        if levels is None:
            levels = out.new_zeros(())
        ctx.mark_non_differentiable(levels)
        return out, levels

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out, _grad_levels):
        x, g, pyr = ctx.saved_tensors
        max_level, min_level, pad_mode, extra, grid_dtype = ctx.cfg
        need_x, need_g = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        lib = _lib.load()
        n, c, hs, ws = x.shape
        ho, wo = g.shape[1], g.shape[2]
        st = _lib.stream()
        go = grad_out.contiguous()
        if go.dtype != x.dtype:
            go = go.to(x.dtype)
        grad_src = torch.zeros(x.shape, dtype=torch.float32, device=x.device) if need_x else None
        grad_pyr = torch.zeros_like(pyr) if (need_x and pyr is not None) else None
        grad_grid = torch.empty(g.shape, dtype=torch.float32, device=x.device) if need_g else None
        scratch = _lib.workspace(lib.gg_mipmap_warp_backward_workspace(n, ho, wo), x.device) if (need_g and extra > 0) else None
        rc = lib.gg_mipmap_warp_backward(_lib.ptr(grad_src), _lib.ptr(grad_pyr), _lib.ptr(grad_grid), _lib.ptr(scratch), go.data_ptr(),
                                         x.data_ptr(), _lib.ptr(pyr), g.data_ptr(), _lib.dtype_code(x), n, c, hs, ws,
                                         ho, wo, extra, max_level, min_level, pad_mode, st)
        _lib.check(rc, "gg_mipmap_warp_backward")
        if need_x and extra > 0:
            rc = lib.gg_mipmap_build_backward(grad_src.data_ptr(), grad_pyr.data_ptr(), n * c, hs, ws, extra, st)
            _lib.check(rc, "gg_mipmap_build_backward")
        if grad_src is not None and grad_src.dtype != x.dtype:
            grad_src = grad_src.to(x.dtype)
        if grad_grid is not None and grad_grid.dtype != grid_dtype:
            grad_grid = grad_grid.to(grid_dtype)
        return grad_src, grad_grid, None, None, None, None


class _StnSample(Function):
    """The STN's sampling in one forward pass (csrc/warp.cu `warp_compose_fwd_kernel`): the sampling grid is generated
    inside the sampler from the head's raw outputs (mode 1: affine matrices; mode 2: low-res flow + convex up-sampling mask
    [+ base warp, alpha]) and written out as a by-product.  Backward = the sampler's backward on the saved grid, then the
    grid generator's (an einsum for the affine case, the flow-composition kernel for the flow case)."""

    @staticmethod
    def forward(ctx, inputs, theta, low, mask, identity, alpha, mode, out_hw, s, max_level, min_level, pad_mode, extra):
        _lib.require_cuda(inputs, theta, low, mask, identity, alpha)
        lib = _lib.load()
        x = inputs.contiguous()
        n, c, hs, ws = x.shape
        ho, wo = out_hw
        code = _lib.dtype_code(x)
        st = _lib.stream()

        def f32(t):
            if t is None:
                return None
            t = t.detach()
            return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()
        th, lo, mk, idn, al = f32(theta), f32(low), f32(mask), f32(identity), f32(alpha)
        lh = lw = 0
        if mode == 2:
            if lo.dim() != 4 or lo.shape[0] != n or lo.shape[-1] != 2:
                raise RuntimeError("stn_sample: low-res flow must be (N, h, w, 2) with N = the image batch")
            lh, lw = lo.shape[1], lo.shape[2]
            if mk.numel() != n * 9 * s * s * lh * lw or idn.numel() != ho * wo * 2:
                raise RuntimeError("stn_sample: mask must be (N, 9*s*s, h, w) and identity_flow (1, s*h, s*w, 2)")
            if al is not None:
                al = al.reshape(-1)
                if al.numel() == 1:
                    al = al.expand(n).contiguous()
                elif al.numel() != n:
                    raise RuntimeError("stn_sample: alpha must have 1 or N elements")
            if th is not None and th.numel() != n * 6:
                raise RuntimeError("stn_sample: base_warp must be (N, 2, 3)")
        elif th is None or th.numel() != n * 6:
            raise RuntimeError("stn_sample: theta must be (N, 2, 3)")
        pyr = None
        if extra > 0:
            elems = lib.gg_mipmap_pyramid_elems(n * c, hs, ws, extra)
            if elems < 0:
                raise RuntimeError("MipmapWarp: a %dx%d source cannot host %d mip levels" % (hs, ws, extra))
            pyr = torch.empty(max(int(elems), 1), dtype=torch.float32, device=x.device)
            _lib.check(lib.gg_mipmap_build(pyr.data_ptr(), x.data_ptr(), code, n * c, hs, ws, extra, st), "gg_mipmap_build")
        out = torch.empty((n, c, ho, wo), dtype=x.dtype, device=x.device)
        grid = torch.empty((n, ho, wo, 2), dtype=torch.float32, device=x.device)
        delta = torch.empty((n, ho, wo, 2), dtype=torch.float32, device=x.device) if mode == 2 else None
        levels = torch.empty((n, ho, wo), dtype=torch.float32, device=x.device) if extra > 0 else None
        rc = lib.gg_stn_sample_forward(out.data_ptr(), grid.data_ptr(), _lib.ptr(delta), _lib.ptr(levels), x.data_ptr(),
                                       _lib.ptr(pyr), _lib.ptr(th), _lib.ptr(lo), _lib.ptr(mk), _lib.ptr(idn), _lib.ptr(al),
                                       mode, code, n, c, hs, ws, ho, wo, lh, lw, s, extra, max_level, min_level, pad_mode, st)
        _lib.check(rc, "gg_stn_sample_forward")
        ctx.save_for_backward(x, grid, pyr, th, lo, mk, idn, al)
        ctx.cfg = (mode, s, max_level, min_level, pad_mode, extra,
                   None if theta is None else (theta.dtype, tuple(theta.shape)),
                   None if low is None else low.dtype, None if mask is None else (mask.dtype, tuple(mask.shape)))
        if delta is None:
            delta = out.new_zeros(())
        if levels is None:
            levels = out.new_zeros(())
        ctx.mark_non_differentiable(levels)
        return out, grid, delta, levels

    @staticmethod
    @once_differentiable
    def backward(ctx, g_out, g_grid, g_delta, _g_levels):
        x, grid, pyr, th, lo, mk, idn, al = ctx.saved_tensors
        mode, s, max_level, min_level, pad_mode, extra, theta_info, low_dt, mask_info = ctx.cfg
        need_x, need_theta, need_low, need_mask = ctx.needs_input_grad[:4]
        lib = _lib.load()
        n, c, hs, ws = x.shape
        ho, wo = grid.shape[1], grid.shape[2]
        st = _lib.stream()
        need_grid = need_theta or need_low or need_mask
        grad_src = torch.zeros(x.shape, dtype=torch.float32, device=x.device) if need_x else None
        grad_pyr = torch.zeros_like(pyr) if (need_x and pyr is not None) else None
        gg = None
        if g_out is not None and (need_x or need_grid):
            go = g_out.contiguous()
            if go.dtype != x.dtype:
                go = go.to(x.dtype)
            gg = torch.empty(grid.shape, dtype=torch.float32, device=x.device) if need_grid else None
            scratch = _lib.workspace(lib.gg_mipmap_warp_backward_workspace(n, ho, wo), x.device) if (need_grid and extra > 0) else None
            rc = lib.gg_mipmap_warp_backward(_lib.ptr(grad_src), _lib.ptr(grad_pyr), _lib.ptr(gg), _lib.ptr(scratch), go.data_ptr(), x.data_ptr(),
                                             _lib.ptr(pyr), grid.data_ptr(), _lib.dtype_code(x), n, c, hs, ws, ho, wo, extra,
                                             max_level, min_level, pad_mode, st)
            _lib.check(rc, "gg_mipmap_warp_backward")
            if need_x and extra > 0:
                _lib.check(lib.gg_mipmap_build_backward(grad_src.data_ptr(), grad_pyr.data_ptr(), n * c, hs, ws, extra, st),
                           "gg_mipmap_build_backward")
        if need_grid and g_grid is not None and g_grid.dim() == 4:     # the caller also used the returned grid
            gg = g_grid.float().contiguous() if gg is None else gg + g_grid.float()
        g_theta = g_low = g_mask = None
        if mode == 1:
            if need_theta and gg is not None:
                # grid = [bx, by, 1] . theta^T  ->  d theta[n, i, k] = sum_yx gg[n, y, x, i] * base[y, x, k]
                bx = (2.0 * torch.arange(wo, device=x.device, dtype=torch.float32) + 1.0) / wo - 1.0
                by = (2.0 * torch.arange(ho, device=x.device, dtype=torch.float32) + 1.0) / ho - 1.0
                g_theta = torch.stack([torch.einsum("nyxi,x->ni", gg, bx), torch.einsum("nyxi,y->ni", gg, by), gg.sum(dim=(1, 2))], dim=2)
                g_theta = g_theta.reshape(theta_info[1]).to(theta_info[0])
        else:
            gd = g_delta.float().contiguous() if (g_delta is not None and g_delta.dim() == 4) else None
            if (need_low or need_mask or need_theta) and (gg is not None or gd is not None):
                g_mask = torch.empty_like(mk) if need_mask else None
                g_low = torch.empty_like(lo) if need_low else None
                g_base = torch.empty((n, 2, 3), dtype=torch.float32, device=x.device) if (need_theta and th is not None) else None
                lh, lw = lo.shape[1], lo.shape[2]
                scratch = _lib.workspace(lib.gg_flow_compose_backward_workspace(n, lh, lw, s), x.device) if (g_low is not None or g_base is not None) else None
                rc = lib.gg_flow_compose_backward(_lib.ptr(g_mask), _lib.ptr(g_low), _lib.ptr(g_base), _lib.ptr(scratch), _lib.ptr(gd), _lib.ptr(gg),
                                                  lo.data_ptr(), mk.data_ptr(), _lib.ptr(idn), _lib.ptr(th), _lib.ptr(al),
                                                  n, lh, lw, s, st)
                _lib.check(rc, "gg_flow_compose_backward")
                if g_mask is not None:
                    g_mask = g_mask.reshape(mask_info[1]).to(mask_info[0])
                if g_low is not None:
                    g_low = g_low.to(low_dt)
                if g_base is not None:
                    g_theta = g_base.reshape(theta_info[1]).to(theta_info[0])
        if grad_src is not None and grad_src.dtype != x.dtype:
            grad_src = grad_src.to(x.dtype)
        return (grad_src, g_theta, g_low, g_mask) + (None,) * 9


def _levels_for(inputs, max_num_levels, min_level):
    max_level = float(max_num_levels) - 1.0
    wanted = int(math.ceil(max(max_level, float(min_level), 0.0)))
    extra = feasible_levels(inputs.shape[2], inputs.shape[3], wanted)
    if extra < wanted:
        max_level = min(max_level, float(extra))
        min_level = min(float(min_level), float(extra))
    return max_level, float(min_level), extra


def stn_sample_affine(inputs, theta, out_hw, max_num_levels=None, min_level=0.0, padding_mode="border"):
    """F.affine_grid(theta, align_corners=False) + [antialiased] bilinear sampling of `inputs`, one pass.
    max_num_levels None: plain `Warp`.  -> (out, grid (N, Ho, Wo, 2), levels or None)."""
    if max_num_levels is None:
        max_level, min_level, extra = 0.0, 0.0, 0
    else:
        max_level, min_level, extra = _levels_for(inputs, max_num_levels, min_level)
    out, grid, _, levels = _StnSample.apply(inputs, theta, None, None, None, None, 1, tuple(out_hw), 1, max_level, min_level,
                                            _pad_code(padding_mode), extra)
    return out, grid, (levels if extra > 0 else None)


def stn_sample_flow(inputs, low, mask, identity_flow, base_warp, alpha, downsample, max_num_levels=None, min_level=0.0,
                    padding_mode="border"):
    """FlowHead's upsample_flow + identity + apply_affine + alpha lerp (warping_heads.py:180-193,239-244,268-277) generated
    inside the [antialiased] sampler, one pass.  -> (out, flow (N, sH, sW, 2), delta_flow (N, sH, sW, 2), levels or None)."""
    if max_num_levels is None:
        max_level, min_level, extra = 0.0, 0.0, 0
    else:
        max_level, min_level, extra = _levels_for(inputs, max_num_levels, min_level)
    ho, wo = low.shape[1] * downsample, low.shape[2] * downsample
    out, grid, delta, levels = _StnSample.apply(inputs, base_warp, low, mask, identity_flow, alpha, 2, (ho, wo), int(downsample),
                                                max_level, min_level, _pad_code(padding_mode), extra)
    return out, grid, delta, (levels if extra > 0 else None)


def sample_indices(grid, source_hw, max_num_levels=8, min_level=0.0, padding_mode="border"):
    """The sampler's integer work for `grid` (N, Ho, Wo, 2) over a source of size `source_hw`: int32 (N, Ho, Wo, 4) =
    (x0, y0, l0, l1) -- north-west bilinear corner after the padding-mode transform and floor / ceil of the level of
    detail, from the device functions the sampling kernels use (gg_warp_sample_indices; for exact parity tests)."""
    _lib.require_cuda(grid)
    hs, ws = int(source_hw[0]), int(source_hw[1])
    max_level = float(max_num_levels) - 1.0
    wanted = int(math.ceil(max(max_level, float(min_level), 0.0)))
    extra = feasible_levels(hs, ws, wanted)
    if extra < wanted:
        max_level, min_level = min(max_level, float(extra)), min(float(min_level), float(extra))
    g = grid.detach().float().contiguous()
    n, ho, wo, _ = g.shape
    out = torch.empty(n, ho, wo, 4, dtype=torch.int32, device=g.device)
    with torch.cuda.device(g.device):
        _lib.check(_lib.load().gg_warp_sample_indices(_lib.ptr(out), _lib.ptr(g), n, hs, ws, ho, wo, max_level, float(min_level),
                                                     _pad_code(padding_mode), _lib.stream()), "warp_sample_indices")
    return out


def _pad_code(padding_mode):
    try:
        return _lib.PAD_MODES[padding_mode]
    except KeyError:
        raise RuntimeError("padding_mode must be 'zeros', 'border' or 'reflection', got %r" % (padding_mode,))


def mipmap_warp(inputs, grid, max_num_levels=8, min_level=0.0, padding_mode="border"):
    """Functional form of MipmapWarp.forward: -> (outputs, levels (N, Ho, Wo) fp32)."""
    max_level = float(max_num_levels) - 1.0
    wanted = int(math.ceil(max(max_level, float(min_level), 0.0)))
    extra = feasible_levels(inputs.shape[2], inputs.shape[3], wanted)
    if extra < wanted:  # tiny source: the reference only fails if such a level is actually selected
        max_level = min(max_level, float(extra))
        min_level = min(float(min_level), float(extra))
    out, levels = _MipmapWarp.apply(inputs, grid, max_level, float(min_level), _pad_code(padding_mode), extra)
    if extra == 0:
        levels = torch.zeros(grid.shape[:3], device=grid.device)
    return out, levels


class _TentDownsample(Function):
    """BilinearDownsample as one gather kernel (csrc/resample.cu); backward = its exact adjoint."""

    @staticmethod
    def forward(ctx, input, taps_h, taps_v, stride):
        _lib.require_cuda(input, taps_h, taps_v)
        x = input.contiguous()
        n, c, h, w = x.shape
        p = stride // 2
        oh, ow = (h + 2 * p - 2 * stride) // stride + 1, (w + 2 * p - 2 * stride) // stride + 1
        out = torch.empty((n, c, max(oh, 0), max(ow, 0)), dtype=x.dtype, device=x.device)
        rc = _lib.load().gg_tent_downsample_forward(out.data_ptr(), x.data_ptr(), taps_h.data_ptr(), taps_v.data_ptr(),
                                                    n, c, h, w, stride, _lib.stream())
        _lib.check(rc, "gg_tent_downsample_forward")
        ctx.save_for_backward(taps_h, taps_v)
        ctx.cfg = (stride, tuple(x.shape))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        taps_h, taps_v = ctx.saved_tensors
        stride, (n, c, h, w) = ctx.cfg
        g = grad_output.contiguous()
        gin = torch.empty((n, c, h, w), dtype=g.dtype, device=g.device)
        rc = _lib.load().gg_tent_downsample_backward(gin.data_ptr(), g.data_ptr(), taps_h.data_ptr(), taps_v.data_ptr(),
                                                     n, c, h, w, stride, _lib.stream())
        _lib.check(rc, "gg_tent_downsample_backward")
        return gin, None, None, None


def bilinear_downsample(input, stride, kernel_horz, kernel_vert):
    """Functional form of BilinearDownsample.forward (reference antialiased_sampling.py:254-256): reflect-pad +
    separable tent filter with stride, as ONE gather kernel (csrc/resample.cu).  Half-precision images are filtered in
    fp32 and cast back; there is no ATen route."""
    _lib.require_cuda(input)
    if input.dim() != 4 or 2 * stride > 32:
        raise RuntimeError("bilinear_downsample: expected a (N, C, H, W) image and stride <= 16, got %s, stride %d" %
                           (tuple(input.shape), stride))
    channels = input.shape[1]
    taps = 2 * stride
    th = kernel_horz.reshape(channels, taps).float().contiguous()
    tv = kernel_vert.reshape(channels, taps).float().contiguous()
    if input.dtype == torch.float32:
        return _TentDownsample.apply(input, th, tv, int(stride))
    return _TentDownsample.apply(input.float(), th, tv, int(stride)).to(input.dtype)


def grid_sample_bilinear(inputs, grid, padding_mode="border"):
    """F.grid_sample(inputs, grid, padding_mode=..., align_corners=False) through the fused kernel (no mip levels)."""
    return _MipmapWarp.apply(inputs, grid, 0.0, 0.0, _pad_code(padding_mode), 0)[0]


def _default_ops():
    from ..opset import cuda_ops
    return cuda_ops()


class Warp(nn.Module):
    """Spatial transform without anti-aliasing (reference antialiased_sampling.py:9-16)."""

    def __init__(self, ops=None):
        super().__init__()
        self.ops = ops

    def forward(self, inputs, grid, padding_mode="border"):
        ops = self.ops if self.ops is not None else _default_ops()
        return ops.grid_sample(inputs, grid, padding_mode)


class MipmapWarp(nn.Module):
    """Spatial transform with mipmap anti-aliasing (reference antialiased_sampling.py:19-60)."""

    def __init__(self, max_num_levels=8, ops=None):
        super().__init__()
        self.ops = ops
        self.max_num_levels = max_num_levels
        f = torch.tensor([1.0, 3.0, 3.0, 1.0])
        f = f[:, None] * f[None, :]
        self.register_buffer("blur_filter", (f / f.sum())[None, None])  # state-dict parity; the kernel hard-codes it
        self._levels = None

    @property
    def levels_map(self):
        """levels / (max_num_levels - 1), as the reference stores after every forward (:59)."""
        if self._levels is None:
            return None
        return self._levels / (self.max_num_levels - 1.0)

    def forward(self, inputs, grid, min_level=0.0, padding_mode="border"):
        ops = self.ops if self.ops is not None else _default_ops()
        out, self._levels = ops.mipmap_warp(inputs, grid, self.max_num_levels, min_level, padding_mode)
        return out

    @staticmethod
    def get_max_coord_distance(coords):
        """Max distance to the four replicate-padded neighbours, each clamped at 1 (reference :62-97);
        provided for API parity (plain tensor ops, not on the hot path)."""
        p = F.pad(coords.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="replicate").permute(0, 2, 3, 1)
        around = (p[:, 1:-1, :-2], p[:, 1:-1, 2:], p[:, :-2, 1:-1], p[:, 2:, 1:-1])
        return torch.stack([((o - coords) ** 2).sum(3).clamp(min=1.0).sqrt() for o in around]).max(dim=0).values


class BilinearDownsample(nn.Module):
    """Reflect-pad + separable tent filter with stride (reference antialiased_sampling.py:241-256).
    Same buffers (`kernel_horz`, `kernel_vert`); on sm_100a one gather kernel (csrc/resample.cu) instead of pad + two
    depthwise convolutions (SURVEY.md 8(f) rank 1)."""

    def __init__(self, stride, channels, ops=None):
        super().__init__()
        self.ops = ops
        self.stride = stride
        self.channels = channels
        ramp = np.arange(1, 2 * stride + 1, 2)
        tent = np.concatenate((ramp, ramp[::-1]))
        tent = torch.Tensor(tent / np.sum(tent))
        self.register_buffer("kernel_horz", tent[None, None, None, :].repeat((channels, 1, 1, 1)))
        self.register_buffer("kernel_vert", tent[None, None, :, None].repeat((channels, 1, 1, 1)))
        self.refl = nn.ReflectionPad2d(int(stride / 2))

    def forward(self, input):
        ops = self.ops if self.ops is not None else _default_ops()
        return ops.bilinear_downsample(input, self.stride, self.kernel_horz, self.kernel_vert)
