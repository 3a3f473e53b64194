"""GPU: the fused training-loop bookkeeping (csrc/optim.cu, SURVEY.md 8(f) rank 3) against its references --
FusedAdamEMA vs torch.optim.Adam (the reference's optimiser, train.py:204-205) + the reference's `accumulate`
(models/__init__.py:19-24) evaluated on the CPU, and the fused total-variation loss vs models/losses/loss.py:4-12."""
import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _reference_tv(delta_flow):     # models/losses/loss.py:4-12, reduce_batch=True
    def dist(a):
        return torch.where(a <= 1.0, 0.5 * a.pow(2), a - 0.5).mean()
    dy = dist((delta_flow[:, :-1] - delta_flow[:, 1:]).abs())
    dx = dist((delta_flow[:, :, :-1] - delta_flow[:, :, 1:]).abs())
    return dx + dy


@pytest.mark.parametrize("shape,scale", [((3, 16, 16, 2), 0.3), ((2, 128, 128, 2), 1.5), ((1, 7, 33, 2), 4.0), ((2, 2, 2, 2), 1.0)])
def test_total_variation_loss_kernel(shape, scale):
    from gangealing_b200.stn.transformer import total_variation_loss
    g = torch.Generator().manual_seed(shape[1])
    f = torch.randn(*shape, generator=g) * scale       # differences on both sides of the Huber knee
    fo = f.clone().requires_grad_(True)
    lo = _reference_tv(fo)
    (go,) = torch.autograd.grad(lo, fo, torch.tensor(2.5))
    fg = f.to(DEV).requires_grad_(True)
    lg = total_variation_loss(fg)
    assert lg.shape == ()
    assert_close(lg, lo, rtol=1e-5, what="tv loss")
    (gg,) = torch.autograd.grad(lg, fg, torch.tensor(2.5, device=DEV))
    assert_close(gg, go, rtol=1e-5, what="tv gradient")
    # per-sample form (forward_with_flip's tie-break) keeps the tensor formulation and agrees with it
    per = total_variation_loss(f.to(DEV), reduce_batch=False)
    assert per.shape == (shape[0],)


def test_fused_adam_ema_matches_torch_adam_and_the_reference_ema():
    from gangealing_b200.training.fused_optim import FusedAdamEMA
    g = torch.Generator().manual_seed(0)
    shapes = [(64, 32, 3, 3), (130,), (7, 5), (256, 64, 1, 1), (3, 70001), (1,)]
    ref_a = [torch.randn(*s, generator=g).requires_grad_(True) for s in shapes[:4]]
    ref_b = [torch.randn(*s, generator=g).requires_grad_(True) for s in shapes[4:]]
    ref_ema = [p.detach().clone() for p in ref_a]
    opt_a = torch.optim.Adam(ref_a, lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    opt_b = torch.optim.Adam(ref_b, lr=1e-2, betas=(0.9, 0.999), eps=1e-8)
    decay = 0.5 ** (32 / 10000)

    def dev(p, cl):
        t = p.detach().to(DEV)
        if cl and t.dim() == 4:
            t = t.contiguous(memory_format=torch.channels_last)     # the Trainer stores 4-D STN weights channels-last
        return t.requires_grad_(True)
    our_a = [dev(p, True) for p in ref_a]
    our_b = [dev(p, False) for p in ref_b]
    our_ema = [p.detach().clone(memory_format=torch.preserve_format) for p in our_a]
    opt = FusedAdamEMA([{"params": our_a, "lr": 1e-3}, {"params": our_b, "lr": 1e-2}], ema_pairs=dict(zip(our_a, our_ema)),
                       ema_decay=decay)
    for it in range(6):
        if it == 3:          # learning-rate schedule: device scalars on our side
            for grp in opt_a.param_groups:
                grp["lr"] = 4e-4
            opt.set_lr(0, 4e-4)
            opt.set_lr(1, torch.tensor(2e-3, device=DEV))
            for grp in opt_b.param_groups:
                grp["lr"] = 2e-3
        for p, q in zip(ref_a + ref_b, our_a + our_b):
            gr = torch.randn(p.shape, generator=g) * (10.0 ** (it - 3))
            p.grad = gr.clone()
            q.grad = gr.to(DEV).contiguous(memory_format=torch.channels_last) if (q.dim() == 4 and q.is_contiguous(memory_format=torch.channels_last)) else gr.to(DEV)
        opt_a.step(); opt_b.step()
        with torch.no_grad():
            for e, p in zip(ref_ema, ref_a):
                e.mul_(decay).add_(p.data, alpha=1 - decay)          # models/__init__.py:23-24
        opt.step()
    for p, q in zip(ref_a + ref_b, our_a + our_b):
        assert_close(q, p, rtol=2e-6, what="parameter %s" % (tuple(p.shape),))
    for e, q in zip(ref_ema, our_ema):
        assert_close(q, e, rtol=2e-6, what="ema")
    # optimiser state carries torch.optim.Adam's keys and values
    st_ref, st_our = opt_a.state[ref_a[0]], opt.state[our_a[0]]
    assert set(st_our.keys()) == {"step", "exp_avg", "exp_avg_sq"}
    assert float(st_our["step"]) == float(st_ref["step"]) == 6.0
    assert_close(st_our["exp_avg"], st_ref["exp_avg"], rtol=2e-6, what="exp_avg")
    assert_close(st_our["exp_avg_sq"], st_ref["exp_avg_sq"], rtol=2e-6, what="exp_avg_sq")
    sd = opt.state_dict()
    assert len(sd["param_groups"]) == 2 and len(sd["state"]) == len(shapes)


def test_fused_adam_ema_is_graph_capturable():
    from gangealing_b200.training.fused_optim import FusedAdamEMA
    p = torch.randn(1000, device=DEV).requires_grad_(True)
    e = p.detach().clone()
    grad = torch.randn(1000, device=DEV)
    p.grad = grad
    opt = FusedAdamEMA([{"params": [p], "lr": 1e-3}], ema_pairs={p: e}, ema_decay=0.9)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        opt.step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        opt.step()
    before = p.detach().clone()
    opt.set_lr(0, 0.0)              # a replay reads the device scalar: lr 0 leaves the parameter untouched
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(p.detach(), before)
    opt.set_lr(0, 1e-2)
    graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(p.detach(), before)
    assert float(opt.state[p]["step"]) == 3.0       # side-stream step + two replays (the capture itself executes nothing)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_multi_tensor_weight_scaling_equals_the_per_layer_products(dtype):
    """op/scaled_weights.WeightScaler (the STN's `weight * scale` products of reference networks.py:121-127,146-149 and their
    backward as a few multi-tensor launches) vs the per-layer ATen products ON THE SAME TRAINER: the scaler learns each layer's
    dtype during the first forward of a step scope (layers then still take their own path) and serves them from the second one
    on, so forward+backward #1 (per-layer) and #2 (multi-tensor) on identical weights, latents and noise must give the same
    loss and the same gradients -- same fp32 multiply, same rounding.  cuDNN is held to its deterministic algorithms for the
    comparison: the split-K weight gradients of the non-deterministic ones differ from run to run by about the tolerance."""
    import contextlib
    from gangealing_b200.training import TrainConfig, Trainer
    cfg = TrainConfig(gen_size=128, flow_size=64, dim_latent=32, n_mlp=2, batch=2, inject=3, gen_channel_multiplier=1,
                      stn_channel_multiplier=0.25, tv_weight=10.0, dtype=dtype)
    tr = Trainer(cfg, DEV)
    sc = tr.weight_scaler
    assert sc is not None and len(sc.by_module) >= 20 and len(sc.groups) >= 1
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():    # leave the zero-initialised identity warp so that every gradient is non-trivial
        for name, prm in tr.t_module.named_parameters():
            if "warp_head" in name:
                prm.copy_((0.05 * torch.randn(prm.shape, generator=g)).to(DEV))
    z = torch.randn(2, 32, generator=g).to(DEV)
    params = list(tr.t_module.parameters())

    def forward_backward(use_scaler):
        torch.manual_seed(100)                    # identical device-side noise draws
        scope = sc.step() if use_scaler else contextlib.nullcontext()
        with scope:
            ld = tr.losses(z)
            for p in params:
                p.grad = None
            (ld["p"] + cfg.tv_weight * ld["tv"]).backward()
        return ld["p"].detach().clone(), [p.grad.detach().clone() for p in params]

    flags = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        l0, g0 = forward_backward(False)          # per-layer products
        _, _ = forward_backward(True)             # scope #1: the scaler only learns the dtypes
        assert all(e.dtype is not None for e in sc.by_module.values())
        assert all(not grp.tables for grp in sc.groups)
        l2, g2 = forward_backward(True)           # scope #2: multi-tensor launches
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = flags
    assert all(len(grp.tables) >= 2 for grp in sc.groups)          # every group launched forward AND backward
    assert all(grp.outputs is None for grp in sc.groups) and not sc.active       # nothing outlives the scope
    tol = 1e-5 if dtype == "f32" else 1e-3
    assert_close(l2, l0, rtol=tol, what="loss")
    flat0, flat2 = torch.cat([t.flatten() for t in g0]), torch.cat([t.flatten() for t in g2])
    assert flat0.abs().max() > 0
    assert_close(flat2, flat0, rtol=tol, what="all STN gradients")
    for a, b, (name, _) in zip(g0, g2, tr.t_module.named_parameters()):
        if a.abs().max() > 0:
            assert_close(b, a, rtol=20 * tol, what=name)
    # whole steps (optimiser included) stay finite, eagerly and from a captured graph
    for _ in range(2):
        out = tr.step(z)
    tr.capture(warmup=2)
    out = tr.step(z)
    assert all(torch.isfinite(v) for v in out.values())
