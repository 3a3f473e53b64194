"""Flow composition of the flow STN head -- one fused kernel per direction (csrc/flow.cu).

`flow_compose(low_res_flow, mask, identity_flow, base_warp, alpha, downsample)` returns
(delta_flow, flow) exactly as reference FlowHead.forward computes them (warping_heads.py:239-244):
RAFT convex upsampling (upsample_flow :180-193), identity + delta, apply_affine (:268-277), alpha lerp.
`apply_affine(matrix, grid)` and `upsample_flow(flow, mask, downsample)` keep the reference call surfaces.
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from .. import _lib


def _f32c(t):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.float().contiguous()
    return t


class _FlowCompose(Function):
    @staticmethod
    def forward(ctx, low, mask, identity, base, alpha, s, want_flow):
        _lib.require_cuda(low, mask, identity, base, alpha)
        if low.dim() != 4 or low.shape[-1] != 2:
            raise RuntimeError("flow_compose: low-res flow must be (N, H, W, 2), got %s" % (tuple(low.shape),))
        n, h, w, _ = low.shape
        if mask.shape[0] != n or mask.numel() != n * 9 * s * s * h * w:
            raise RuntimeError("flow_compose: mask must be (N, 9*%d*%d, H, W), got %s" % (s, s, tuple(mask.shape)))
        low_c, mask_c, ident_c, base_c, alpha_c = _f32c(low), _f32c(mask), _f32c(identity), _f32c(base), _f32c(alpha)
        if ident_c is not None and ident_c.numel() != s * h * s * w * 2:
            raise RuntimeError("flow_compose: identity_flow must be (1, %d, %d, 2)" % (s * h, s * w))
        if base_c is not None and base_c.numel() != n * 6:
            raise RuntimeError("flow_compose: base_warp must be (N, 2, 3)")
        if alpha_c is not None:
            # the reference broadcasts `identity_flow.lerp(flow, alpha[:, None, None, None])` (warping_heads.py:243-244):
            # a 1-element alpha serves any batch; the kernel reads alpha[n] for every n, so expand it here
            alpha_c = alpha_c.reshape(-1)
            if alpha_c.numel() == 1:
                alpha_c = alpha_c.expand(n).contiguous()
            elif alpha_c.numel() != n:
                raise RuntimeError("flow_compose: alpha must have 1 or N=%d elements, got %d" % (n, alpha_c.numel()))
        delta = torch.empty((n, s * h, s * w, 2), dtype=torch.float32, device=low.device)
        flow = torch.empty_like(delta) if want_flow else None
        rc = _lib.load().gg_flow_compose_forward(delta.data_ptr(), _lib.ptr(flow), low_c.data_ptr(), mask_c.data_ptr(),
                                                 _lib.ptr(ident_c), _lib.ptr(base_c), _lib.ptr(alpha_c), n, h, w, s,
                                                 _lib.stream())
        _lib.check(rc, "gg_flow_compose_forward")
        ctx.save_for_backward(low_c, mask_c, ident_c, base_c, alpha_c)
        ctx.cfg = (s, low.dtype, mask.dtype, None if base is None else (base.dtype, tuple(base.shape)), tuple(mask.shape))
        if flow is None:
            flow = delta.new_zeros(())
            ctx.mark_non_differentiable(flow)
        return delta, flow

    @staticmethod
    @once_differentiable
    def backward(ctx, g_delta, g_flow):
        low, mask, ident, base, alpha = ctx.saved_tensors
        s, low_dt, mask_dt, base_info, mask_shape = ctx.cfg
        n, h, w, _ = low.shape
        need_low, need_mask, _, need_base = ctx.needs_input_grad[:4]
        g_delta = _f32c(g_delta) if g_delta is not None else None
        g_flow = _f32c(g_flow) if (g_flow is not None and g_flow.dim() == 4) else None
        g_mask = torch.empty_like(mask) if need_mask else None
        g_low = torch.empty_like(low) if need_low else None
        g_base = torch.empty((n, 2, 3), dtype=torch.float32, device=low.device) if (need_base and base is not None) else None
        scratch = _lib.workspace(_lib.load().gg_flow_compose_backward_workspace(n, h, w, s), low.device) if (g_low is not None or g_base is not None) else None
        rc = _lib.load().gg_flow_compose_backward(_lib.ptr(g_mask), _lib.ptr(g_low), _lib.ptr(g_base), _lib.ptr(scratch), _lib.ptr(g_delta),
                                                  _lib.ptr(g_flow), low.data_ptr(), mask.data_ptr(), _lib.ptr(ident),
                                                  _lib.ptr(base), _lib.ptr(alpha), n, h, w, s, _lib.stream())
        _lib.check(rc, "gg_flow_compose_backward")
        if g_mask is not None:
            g_mask = g_mask.reshape(mask_shape).to(mask_dt)
        if g_low is not None:
            g_low = g_low.to(low_dt)
        if g_base is not None:
            g_base = g_base.reshape(base_info[1]).to(base_info[0])
        return g_low, g_mask, None, g_base, None, None, None


def flow_compose(low_res_flow, mask, identity_flow, base_warp=None, alpha=None, downsample=8):
    """-> (delta_flow (N, sH, sW, 2), flow (N, sH, sW, 2)); fp32."""
    return _FlowCompose.apply(low_res_flow, mask, identity_flow, base_warp, alpha, downsample, True)


def upsample_flow(flow, mask, downsample=8):
    """RAFT convex upsampling [H/s, W/s, 2] -> [H, W, 2] (reference FlowHead.upsample_flow)."""
    return _FlowCompose.apply(flow, mask, None, None, None, downsample, False)[0]


def apply_affine(matrix, grid):
    """[gx, gy, 1] @ matrix^T at every grid point (reference warping_heads.py:268-277); plain tensor ops --
    inside the flow head this step is fused into flow_compose."""
    n = grid.size(0)
    flat = grid.reshape(n, -1, 2)
    out = flat @ matrix[:, :, :2].transpose(1, 2) + matrix[:, None, :, 2]
    return out.reshape(grid.size())
