"""GPU: this repo's kernels against the REFERENCE'S OWN CUDA KERNELS recompiled for sm_100a (oracle/_ref/*.so, built by
oracle/build_ref.py from models/stylegan2/op/upfirdn2d_kernel.cu:209-369 and fused_bias_act_kernel.cu:52-99 where they
lie) on identical device inputs -- the comparison north_star words ("outputs match the reference's own kernels on
identical latents/inputs within 1e-3 relative fp32").  Includes the generator's full-size 257^2 -> 256^2 layer in both
activation layouts, and the CPU oracle against the same reference kernels (pins the restatement to the CUDA code too).
What the reference kernels computed is kept in tests/golden/reference_kernels.npz (conftest.Pinned: a seeded sample of each
output; GG_RECORD_GOLDEN=1 with oracle/_ref/ built recomputes it on the GPU).
"""
import pytest
import torch

from conftest import Pinned, assert_close
from oracle import build_ref
from oracle import stylegan2_ops as so

pytestmark = pytest.mark.gpu
DEV = "cuda"
CL = torch.channels_last


@pytest.fixture(scope="module")
def pin():
    p = Pinned("reference_kernels")
    yield p
    p.save()


def _load(name):
    mod = build_ref.load_ref(name)
    assert mod is not None, "oracle/_ref/%s.so not built (python -m oracle.build_ref)" % name
    return mod


def ref_upfirdn2d(x, k, up=1, down=1, pad=(0, 0)):      # the reference's Python wrapper, op/upfirdn2d.py:88-124
    n, c, h, w = x.shape
    out = _load("upfirdn2d_ref").upfirdn2d(x.reshape(-1, h, w, 1).contiguous(), k.contiguous(), up, up, down, down, pad[0], pad[1],
                                           pad[0], pad[1])
    return out.view(n, c, out.shape[1], out.shape[2])


def ref_fused_bias_act(*args):
    return _load("fused_ref").fused_bias_act(*args)


def _k1331(gain=1.0):
    return (so.make_kernel([1, 3, 3, 1]) * gain).to(DEV)


@pytest.mark.parametrize("shape,up,down,pad,gain", [
    ((2, 128, 257, 257), 1, 1, (1, 1), 4.0),     # generator blur, 256^2 layer (full size)
    ((2, 512, 65, 65), 1, 1, (1, 1), 4.0),       # generator blur, 64^2 layer
    ((3, 512, 9, 9), 1, 1, (1, 1), 4.0),         # generator blur, 8^2 layer
    ((2, 64, 128, 128), 1, 1, (2, 2), 1.0),      # STN ResBlock conv2 blur
    ((2, 64, 128, 128), 1, 1, (1, 1), 1.0),      # STN ResBlock skip blur
    ((2, 3, 128, 128), 2, 1, (2, 1), 4.0),       # to-RGB skip upsample
    ((2, 3, 256, 256), 1, 2, (1, 1), 1.0),       # its backward (down 2)
    ((1, 5, 31, 47), 1, 1, (-1, 2), 1.0),        # negative pad (crop), odd sizes
])
def test_upfirdn2d_equals_the_reference_cuda_kernel(pin, shape, up, down, pad, gain):
    from gangealing_b200 import op
    g = torch.Generator().manual_seed(shape[1] + shape[2])
    x = torch.randn(*shape, generator=g).to(DEV)
    k = _k1331(gain)
    got = {"NCHW kernel": op.upfirdn2d(x, k, up=up, down=down, pad=pad)}
    if shape[1] % 32 == 0 and up == 1 and down == 1:
        got["channels-last (TMA tensor-map) kernel"] = op.upfirdn2d(x.contiguous(memory_format=CL), k, pad=pad)
        assert got["channels-last (TMA tensor-map) kernel"].is_contiguous(memory_format=CL)
    if x.numel() <= 4_000_000:
        got["CPU oracle"] = so.upfirdn2d_ref(x.cpu(), k.cpu(), up=up, down=down, pad=pad)
        assert_close(got["NCHW kernel"], got["CPU oracle"], rtol=1e-5, what="NCHW kernel vs CPU oracle, every element")
    pairs = pin("upfirdn2d%s" % ((shape, up, down, pad, gain),), tuple(got.values()),
                lambda: (ref_upfirdn2d(x, k, up, down, pad),) * len(got))
    for what, (a, expect) in zip(got, pairs):
        assert_close(a, expect, rtol=1e-5, what=what)


def test_upfirdn2d_generic_filter_equals_the_reference_cuda_kernel(pin):
    from gangealing_b200 import op
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 32, 40, 52, generator=g).to(DEV)
    k = torch.randn(4, 3, generator=g).to(DEV)       # not symmetric, not rank-1-tested: true convolution (flipped taps)
    got = (op.upfirdn2d(x, k, pad=(2, 1)), op.upfirdn2d(x.contiguous(memory_format=CL), k, pad=(2, 1)))
    for what, (a, expect) in zip(("NCHW", "NHWC"), pin("generic_filter", got, lambda: (ref_upfirdn2d(x, k, 1, 1, (2, 1)),) * 2)):
        assert_close(a, expect, rtol=1e-5, what=what)


@pytest.mark.parametrize("shape,up,down,pad", [((2, 3, 64, 64), 2, 1, (2, 1)), ((3, 3, 4, 4), 2, 1, (2, 1)), ((1, 3, 6, 10), 2, 1, (2, 1)),
                                               ((2, 3, 128, 128), 1, 2, (1, 1)), ((3, 3, 8, 8), 1, 2, (1, 1)), ((1, 2, 12, 20), 1, 2, (1, 1)),
                                               ((1, 3, 7, 9), 2, 1, (2, 1)), ((1, 3, 10, 10), 1, 2, (1, 1))])   # last two: generic path
def test_upfirdn2d_x2_resamplers_with_an_asymmetric_filter(pin, shape, up, down, pad):
    """The polyphase x2 up-sampler / decimator (to-RGB skip and its backward) with a NON-symmetric 4x4 filter: tap flipping
    and phase selection must follow the reference kernel (upfirdn2d_kernel.cu:137), exactly as the generic path does."""
    from gangealing_b200 import op
    g = torch.Generator().manual_seed(shape[2] * 7 + up)
    x = torch.randn(*shape, generator=g).to(DEV)
    k = torch.randn(4, 4, generator=g).to(DEV)
    got = (op.upfirdn2d(x, k, up=up, down=down, pad=pad), so.upfirdn2d_ref(x.cpu(), k.cpu(), up=up, down=down, pad=pad))
    assert_close(got[0], got[1], rtol=1e-5, what="kernel vs CPU oracle, every element")
    pairs = pin("x2%s" % ((shape, up, down, pad),), got, lambda: (ref_upfirdn2d(x, k, up, down, pad),) * 2)
    for what, (a, expect) in zip(("kernel vs reference CUDA", "CPU oracle"), pairs):
        assert_close(a, expect, rtol=1e-5, what=what)


@pytest.mark.parametrize("shape", [(2, 128, 256, 256), (4, 512, 64, 64), (3, 512), (2, 64, 33, 31)])
def test_fused_bias_act_forward_and_backward_equal_the_reference_cuda_kernel(pin, shape):
    from gangealing_b200 import op
    g = torch.Generator().manual_seed(len(shape) + shape[1])
    x = torch.randn(*shape, generator=g).to(DEV)
    b = torch.randn(shape[1], generator=g).to(DEV)
    go = torch.randn(*shape, generator=g).to(DEV)

    def reference():
        empty = x.new_empty(0)
        out_ref = ref_fused_bias_act(x, b, empty, 3, 0, 0.2, 2 ** 0.5)               # fused_act.py:55
        gx_ref = ref_fused_bias_act(go, empty, out_ref, 3, 1, 0.2, 2 ** 0.5)          # fused_act.py:29-31
        gb_ref = gx_ref.sum([0] + list(range(2, x.dim())))                            # fused_act.py:33-38
        return (out_ref, gx_ref, gb_ref) * len(layouts)
    layouts = ("nchw", "nhwc") if x.dim() == 4 and shape[1] % 4 == 0 else ("nchw",)
    got = []
    for layout in layouts:
        xi = (x.contiguous(memory_format=CL) if layout == "nhwc" else x.clone()).requires_grad_(True)
        bi = b.clone().requires_grad_(True)
        out = op.fused_leaky_relu(xi, bi, 0.2, 2 ** 0.5)
        gx, gb = torch.autograd.grad(out, (xi, bi), go.contiguous(memory_format=CL) if layout == "nhwc" else go)
        got += [out, gx, gb]
    pairs = pin("fused_bias_act%s" % (shape,), got, reference)
    for i, layout in enumerate(layouts):
        (out, out_ref), (gx, gx_ref), (gb, gb_ref) = pairs[3 * i:3 * i + 3]
        # the same fp32 expression (x + b, select, one multiply) in both kernels: agreement to the last bit or two
        assert_close(out, out_ref, rtol=5e-7, what=layout + " forward")
        assert_close(gx, gx_ref, rtol=5e-7, what=layout + " grad input")
        assert_close(gb, gb_ref, rtol=1e-4, what=layout + " bias gradient (summation order differs)")


def test_fused_tail_equals_the_reference_kernel_sequence_at_full_size(pin):
    """The fused blur+noise+bias+lrelu tail (the roofline kernel) at the benchmark's 257^2 -> 256^2 shape against the
    reference's three-kernel sequence Blur -> NoiseInjection -> FusedLeakyReLU (networks.py:266,291-298,346-348) run with
    the reference's own CUDA kernels.  Leaky-ReLU flips slope where the pre-activation is within rounding of 0, so the
    comparison is made (a) on the linear pre-activation (act=identity via slope 1) everywhere and (b) on the activated
    output wherever |pre-activation| exceeds the rounding noise."""
    from gangealing_b200 import op
    g = torch.Generator().manual_seed(11)
    n, c, h = 2, 128, 257
    x = torch.randn(n, c, h, h, generator=g).to(DEV)
    noise = torch.randn(n, 1, h - 1, h - 1, generator=g).to(DEV)
    nw = torch.tensor([0.37], device=DEV)
    b = torch.randn(c, generator=g).to(DEV)
    k = _k1331(4.0)
    got = []
    for layout in ("nchw", "nhwc"):
        xi = x.contiguous(memory_format=CL) if layout == "nhwc" else x
        got += [op.blur_noise_bias_act(xi, k, (1, 1), noise, nw, b, negative_slope=1.0),
                op.blur_noise_bias_act(xi, k, (1, 1), noise, nw, b, negative_slope=0.2)]
    ref = {}

    def reference():      # the activated output is kept only where the REFERENCE's pre-activation is safe (NaN elsewhere)
        if not ref:
            empty = x.new_empty(0)
            pre = ref_upfirdn2d(x, k, 1, 1, (1, 1)) + nw * noise
            safe = (pre + b.view(1, -1, 1, 1)).abs() > 1e-4
            act_ref = ref_fused_bias_act(pre, b, empty, 3, 0, 0.2, 2 ** 0.5)
            ref.update(lin=ref_fused_bias_act(pre, b, empty, 3, 0, 1.0, 2 ** 0.5),      # slope 1: linear
                       act=torch.where(safe, act_ref, torch.full_like(act_ref, float("nan"))), safe=safe.float().mean().item())
        return (ref["lin"], ref["act"]) * 2
    def safe_fraction():
        reference()
        return ref["safe"]
    assert float(pin.value("fused_tail.safe_fraction", safe_fraction)) > 0.999
    pairs = pin("fused_tail", got, reference, keep=1 << 10)
    for i, layout in enumerate(("nchw", "nhwc")):
        (lin, lin_ref), (act, act_ref) = pairs[2 * i:2 * i + 2]
        assert_close(lin, lin_ref, rtol=5e-6, what=layout + " pre-activation")
        safe = torch.isfinite(act_ref)
        assert safe.any()
        err = (act[safe] - act_ref[safe]).abs().max().item()
        assert err <= 5e-6 * act_ref[safe].abs().max().item(), (layout, err)
