"""Perceptual-loss front end (SURVEY.md 8(f) rank 2): oracle vs the reference-generated fixture (CPU), the fused
channels-last kernels vs the oracle through the C ABI (GPU)."""
import pytest
import torch

from conftest import Pinned, assert_close, golden_cases, load_golden, state_dict_layout, zeros_state_dict
from oracle.perceptual import feature_distance_ref

DEV = "cuda"


def _case(blob, name):
    w = blob.get(name + ".weight")
    return blob[name + ".f0"], blob[name + ".f1"], w, blob[name + ".out"], blob[name + ".gout"], blob[name + ".g0"], blob[name + ".g1"]


def test_oracle_matches_reference_fixture():
    blob = load_golden("perceptual")
    names = golden_cases(blob)
    assert len(names) >= 5
    for name in names:
        f0, f1, w, out, gout, g0, g1 = _case(blob, name)
        a, b = f0.clone().requires_grad_(True), f1.clone().requires_grad_(True)
        res = feature_distance_ref(a, b, w)
        assert res.shape == out.shape
        assert_close(res, out, rtol=1e-6, what=name + " out")
        ga, gb = torch.autograd.grad(res, [a, b], gout)
        assert_close(torch.nan_to_num(ga, nan=0.0), g0, rtol=1e-6, what=name + " g0")
        assert_close(gb, g1, rtol=1e-6, what=name + " g1")


def test_the_op_refuses_cpu_tensors_and_has_no_eager_route():
    from gangealing_b200.op import feature_distance as mod
    g = torch.Generator().manual_seed(2)
    a, b = torch.rand(2, 12, 5, 5, generator=g), torch.rand(2, 12, 5, 5, generator=g)
    with pytest.raises(RuntimeError):
        mod.feature_distance(a, b, torch.rand(12, generator=g))                           # no CPU path in the product
    assert not hasattr(mod, "_composite")                                                 # and no tensor-op fallback
    assert mod._channels_ok(64) and mod._channels_ok(512) and mod._channels_ok(16) and not mod._channels_ok(12)


def test_perceptual_module_is_key_compatible_with_the_reference_lpips():
    """Reference LPIPS checkpoints (`scaling_layer.*`, `net.slice{k}.{torchvision index}.*`, `lin{k}.model.1.weight`) and
    torchvision VGG16 `features` checkpoints (lpips_backbones.py:103-105) load into the mirror."""
    from gangealing_b200.training.perceptual import PerceptualLoss, get_perceptual_loss
    base = PerceptualLoss()
    keys = set(base.state_dict().keys())
    conv_idx = {1: (0, 2), 2: (5, 7), 3: (10, 12, 14), 4: (17, 19, 21), 5: (24, 26, 28)}
    want = {"scaling_layer.shift", "scaling_layer.scale"}
    for k, idxs in conv_idx.items():
        for i in idxs:
            want |= {"net.slice%d.%d.weight" % (k, i), "net.slice%d.%d.bias" % (k, i)}
    assert keys == want
    lp = PerceptualLoss(divisor=1.0, lpips=True)
    assert {"lin%d.model.1.weight" % k for k in range(5)} <= set(lp.state_dict().keys())
    # a torchvision-style features state dict loads strictly and lands in the right slices
    g = torch.Generator().manual_seed(0)
    feats = {}
    for k, idxs in conv_idx.items():
        for i in idxs:
            w = dict(getattr(base.net, "slice%d" % k).named_children())[str(i)].weight
            feats["%d.weight" % i] = torch.randn(w.shape, generator=g)
            feats["%d.bias" % i] = torch.randn(w.shape[0], generator=g)
    loaded = PerceptualLoss(pretrained_weights=feats)
    assert torch.equal(loaded.state_dict()["net.slice3.12.weight"], feats["12.weight"])
    with pytest.raises(RuntimeError):
        PerceptualLoss(pretrained_weights=dict(feats, **{"30.weight": torch.zeros(1)}))    # strict, like the reference
    assert get_perceptual_loss("cpu", kind="lpips").lpips


def test_reference_lpips_state_dict_loads_into_the_mirror():
    """The layout of the reference LPIPS state dict is kept in tests/golden/state_dicts_lpips.npz (conftest.Pinned)."""
    from gangealing_b200.training.perceptual import PerceptualLoss
    pin = Pinned("state_dicts_lpips")

    def reference(lpips):
        from oracle import refimport
        refimport.import_reference()
        import models.losses.lpips as L
        return state_dict_layout(L.LPIPS(net="vgg", lpips=lpips, pnet_rand=True, pretrained=False, verbose=False))
    for lpips in (False, True):
        layout = pin.value("lpips%d" % lpips, lambda: reference(lpips))
        ours = PerceptualLoss(lpips=lpips)
        missing, unexpected = ours.load_state_dict(zeros_state_dict(layout), strict=False)
        assert not missing and not unexpected, (missing, unexpected)
    pin.save()


@pytest.mark.gpu
def test_fused_kernels_match_reference_fixture():
    from gangealing_b200.op.feature_distance import feature_distance
    blob = load_golden("perceptual")
    for name in golden_cases(blob):
        f0, f1, w, out, gout, g0, g1 = _case(blob, name)
        a = f0.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        b = f1.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        res = feature_distance(a, b, None if w is None else w.to(DEV))
        assert_close(res, out, rtol=1e-5, what=name + " out")
        ga, gb = torch.autograd.grad(res, [a, b], gout.to(DEV))
        assert ga.is_contiguous(memory_format=torch.channels_last)
        assert_close(ga, g0, rtol=1e-4, what=name + " g0")
        assert_close(gb, g1, rtol=1e-4, what=name + " g1")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 64, 64, 64), (2, 128, 33, 31), (3, 256, 16, 16), (2, 512, 8, 8), (1, 512, 1, 1),
                                   (2, 16, 9, 9)])
def test_fused_kernels_match_oracle(shape):
    from gangealing_b200.op.feature_distance import feature_distance
    g = torch.Generator().manual_seed(shape[1] + shape[2])
    f0 = torch.relu(torch.randn(*shape, generator=g))
    f1 = torch.relu(torch.randn(*shape, generator=g) + 0.2)
    go = torch.randn(shape[0], 1, 1, 1, generator=g)
    a, b = f0.clone().requires_grad_(True), f1.clone().requires_grad_(True)
    ro = feature_distance_ref(a, b)
    gao, gbo = torch.autograd.grad(ro, [a, b], go)
    x = f0.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = f1.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    r = feature_distance(x, y)
    assert_close(r, ro, rtol=1e-5, what="out")
    gx, gy = torch.autograd.grad(r, [x, y], go.to(DEV))
    assert_close(gx, gao, rtol=1e-4, what="g0")
    assert_close(gy, gbo, rtol=1e-4, what="g1")
    # symmetry and identity: d(a, b) == d(b, a), d(a, a) == 0 -- size-independent properties
    assert_close(feature_distance(y, x), r, rtol=1e-6)
    assert float(feature_distance(x, x).abs().max()) < 1e-12   # a*ia - b*ib contracts to an fma: one rounding residual
    # planar (NCHW) and half-precision maps are converted to the kernel's layout, never evaluated with tensor ops
    assert_close(feature_distance(f0.to(DEV), f1.to(DEV)), ro, rtol=1e-5, what="NCHW input")
    assert_close(feature_distance(x.detach().bfloat16(), y.detach().bfloat16()),
                 feature_distance_ref(f0.bfloat16().float(), f1.bfloat16().float()), rtol=1e-5, what="bf16 input")


def test_whole_perceptual_loss_matches_the_reference_lpips_fixture():
    """PerceptualLoss (this repo's mirror of LPIPS(net='vgg', lpips=False, pnet_rand=True)/18, lpips.py:13-17) against
    the reference class run with the same seeded VGG16 weights: scaling layer, slice boundaries, distance, gradients."""
    from gangealing_b200.training.perceptual import PerceptualLoss
    from oracle import opset
    blob = load_golden("perceptual_loss")
    loss = opset.fill_convs_in_order(PerceptualLoss(ops=opset.cpu_ops()), 4242)
    in0 = blob["in0"].clone().requires_grad_(True)
    in1 = blob["in1"].clone().requires_grad_(True)
    val = loss(in0, in1)
    assert val.shape == blob["val"].shape
    assert_close(val, blob["val"], rtol=1e-5, what="perceptual distance")
    g0, g1 = torch.autograd.grad(val.sum(), [in0, in1])
    assert_close(g0, blob["g0"], rtol=1e-4, what="d/d in0")
    assert_close(g1, blob["g1"], rtol=1e-4, what="d/d in1")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,shape", [(torch.float32, (2, 64, 32, 32)), (torch.float32, (3, 128, 6, 10)), (torch.float32, (1, 512, 2, 2)),
                                         (torch.bfloat16, (2, 64, 32, 32)), (torch.bfloat16, (2, 256, 8, 4))])
@pytest.mark.parametrize("ties", [False, True])
def test_bias_relu_pool_matches_the_aten_sequence_of_the_reference_backbone(dtype, shape, ties):
    """VGG slice boundary (Conv2d -> ReLU -> [tap] -> MaxPool2d(2,2), lpips_backbones.py:106-121) in one pass each way vs the
    ATen sequence on the CPU.  `ties`: small-integer data, so windows hold EQUAL maxima -- the gradient must go to the first
    one in row-major order (max_pool2d's rule) -- and exact zeros after the ReLU; every value is exactly representable, so
    forward, pooled map and gradients must then be BIT-EXACT."""
    from gangealing_b200.op.vgg_pool import bias_relu_pool
    from oracle.perceptual import bias_relu_pool_ref
    g = torch.Generator().manual_seed(shape[1] + shape[2] + int(ties))
    n, c, h, w = shape
    if ties:
        raw = torch.randint(-3, 4, shape, generator=g).float()
        bias = torch.randint(-1, 2, (c,), generator=g).float()
        gy = torch.randint(-4, 5, shape, generator=g).float()
        gp = torch.randint(-4, 5, (n, c, h // 2, w // 2), generator=g).float()
    else:
        raw, bias = torch.randn(shape, generator=g), torch.randn(c, generator=g)
        gy, gp = torch.randn(shape, generator=g), torch.randn(n, c, h // 2, w // 2, generator=g)
    raw, gy, gp = raw.to(dtype), gy.to(dtype), gp.to(dtype)        # bf16 inputs are the rounded values on both sides
    a = raw.clone().requires_grad_(True)
    y_ref, p_ref = bias_relu_pool_ref(a.float() if dtype == torch.bfloat16 else a, bias)
    if dtype == torch.bfloat16:   # the backbone stores bf16 feature maps: the pool reads the ROUNDED activation
        y_ref = y_ref.to(dtype).float()
        p_ref = torch.nn.functional.max_pool2d(y_ref, 2, 2)
    b = raw.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y, p = bias_relu_pool(b, bias.to(DEV))
    assert y.dtype == dtype and p.dtype == dtype and y.is_contiguous(memory_format=torch.channels_last)
    exact = ties or dtype == torch.float32
    if exact:
        assert torch.equal(y.float().cpu(), y_ref.detach().float()) and torch.equal(p.float().cpu(), p_ref.detach().float())
    else:
        assert_close(y.float(), y_ref, rtol=8e-3, what="relu(raw + bias)")
        assert_close(p.float(), p_ref, rtol=8e-3, what="pooled")
    (ga,) = torch.autograd.grad([y_ref, p_ref], [a], [gy.float(), gp.float()]) if dtype == torch.float32 else (None,)
    (gb,) = torch.autograd.grad([y, p], [b], [gy.to(DEV), gp.to(DEV)])
    if dtype == torch.float32:
        if ties:
            assert torch.equal(gb.cpu(), ga)
        assert_close(gb, ga, rtol=1e-6, what="gradient")
    elif ties:    # bf16 with integers: reference gradient from the fp32 graph of the same (exact) values
        a32 = raw.float().clone().requires_grad_(True)
        y32, p32 = bias_relu_pool_ref(a32, bias)
        (g32,) = torch.autograd.grad([y32, p32], [a32], [gy.float(), gp.float()])
        assert torch.equal(gb.float().cpu(), g32)
    # only one of the two gradients arriving (the other branch unused)
    (g_only_pool,) = torch.autograd.grad(bias_relu_pool(b, bias.to(DEV))[1], [b], [gp.to(DEV)])
    a2 = raw.float().clone().requires_grad_(True)
    (g_ref_pool,) = torch.autograd.grad(bias_relu_pool_ref(a2, bias)[1] if dtype == torch.float32 else
                                        torch.nn.functional.max_pool2d(torch.relu(a2 + bias.reshape(1, -1, 1, 1)), 2, 2), [a2], [gp.float()])
    if exact:
        assert_close(g_only_pool.float(), g_ref_pool, rtol=1e-6, what="pool-only gradient")


@pytest.mark.gpu
def test_bias_relu_pool_argument_checks():
    from gangealing_b200.op.vgg_pool import bias_relu_pool, supported
    x = torch.randn(1, 64, 5, 4, device=DEV)
    assert not supported(x) and supported(torch.randn(1, 64, 4, 4, device=DEV)) and not supported(torch.randn(1, 6, 4, 4, device=DEV))
    with pytest.raises(RuntimeError):
        bias_relu_pool(x, None)
    with pytest.raises(RuntimeError):
        bias_relu_pool(torch.randn(1, 64, 4, 4), None)      # no CPU path


@pytest.mark.gpu
def test_stacked_feature_distance_matches_reference_fixture():
    """feature_distance_stacked(cat(f0, f1)) -- both images' features from ONE backbone pass -- against the reference-generated
    fixture: value and the gradient of BOTH halves, written into one stacked tensor."""
    from gangealing_b200.op.feature_distance import feature_distance_stacked
    blob = load_golden("perceptual")
    for name in golden_cases(blob):
        f0, f1, w, out, gout, g0, g1 = _case(blob, name)
        f = torch.cat([f0, f1], 0).to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        res = feature_distance_stacked(f, None if w is None else w.to(DEV))
        assert_close(res, out, rtol=1e-5, what=name + " out")
        (gf,) = torch.autograd.grad(res, [f], gout.to(DEV))
        n = f0.shape[0]
        assert_close(gf[:n], g0, rtol=1e-4, what=name + " g0")
        assert_close(gf[n:], g1, rtol=1e-4, what=name + " g1")


@pytest.mark.gpu
def test_whole_perceptual_loss_on_the_gpu_matches_the_reference_lpips_fixture():
    """The product path of the perceptual loss (one stacked VGG16 pass on cuDNN, fused bias+ReLU(+pool) passes, stacked distance
    kernel) against the reference LPIPS class run on the CPU with the same seeded weights: value and both input gradients."""
    from gangealing_b200.training.perceptual import PerceptualLoss
    from oracle import opset
    blob = load_golden("perceptual_loss")
    loss = opset.fill_convs_in_order(PerceptualLoss(), 4242).to(DEV).to(memory_format=torch.channels_last)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        in0 = blob["in0"].to(DEV).requires_grad_(True)
        in1 = blob["in1"].to(DEV).requires_grad_(True)
        val = loss(in0, in1) / 1.0
        assert_close(val, blob["val"], rtol=1e-4, what="loss value")
        g0, g1 = torch.autograd.grad(val.sum(), [in0, in1])
        assert_close(g0, blob["g0"], rtol=2e-4, what="gradient wrt image 0")
        assert_close(g1, blob["g1"], rtol=2e-4, what="gradient wrt image 1")
    finally:
        torch.backends.cudnn.allow_tf32 = old
