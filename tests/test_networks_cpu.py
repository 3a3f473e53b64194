"""CPU: the host-side networks (run on the oracle op set) against (a) the reference's own modules when the
checkout is present in this container and (b) fixtures generated from them -- state-dict compatibility included."""

import pytest
import torch

from conftest import Pinned, assert_close, load_golden, state_dict_layout, zeros_state_dict
from oracle import opset, refimport

CPU = opset.cpu_ops()


def _gen(ops=CPU):
    from gangealing_b200.stylegan2 import Generator
    return Generator(32, 32, 2, channel_multiplier=2, ops=ops).eval()


def _stn(transforms, ops=CPU):
    from gangealing_b200.stn import get_stn
    return get_stn(list(transforms), flow_size=64, supersize=128, channel_multiplier=0.5, num_heads=1, ops=ops).eval()


def test_generator_matches_reference_fixture():
    blob = load_golden("networks")
    g = opset.fill_parameters(_gen(), 1)
    noise = [blob["gen.noise%d" % i] for i in range(g.num_layers)]
    with torch.no_grad():
        img, lat = g([blob["gen.z"]], noise=noise, return_latents=True)
        img2, _ = g([lat], input_is_latent=True, noise=noise)
    assert_close(img, blob["gen.image"], rtol=1e-5, what="G image")
    assert_close(lat, blob["gen.latent"], rtol=1e-6, what="G latent")
    assert_close(img2, blob["gen.image"], rtol=1e-5, what="G from latent")


@pytest.mark.parametrize("transforms", [("similarity",), ("similarity", "flow")])
def test_stn_matches_reference_fixture(transforms):
    blob = load_golden("networks")
    tag = "stn_" + "_".join(transforms)
    stn = opset.fill_parameters(_stn(transforms), 3, gain=0.3)
    with torch.no_grad():
        out, grid, fm = stn(blob[tag + ".x"], return_warp=True, return_flow=True, padding_mode="reflection")
    assert_close(out, blob[tag + ".out"], rtol=1e-4, what="STN out")
    assert_close(grid, blob[tag + ".grid"], rtol=1e-5, what="STN grid")
    assert_close(fm, blob[tag + ".fm"], rtol=1e-5, what="STN flow/matrix")


def test_config1_similarity_stn_64_cpu():
    """BASELINE config 1: similarity-only STN, 64x64 synthetic batch on CPU, three padding modes."""
    blob = load_golden("networks")
    from gangealing_b200.stn import get_stn
    stn = get_stn(["similarity"], flow_size=64, supersize=64, channel_multiplier=0.5, num_heads=1, ops=CPU).eval()
    opset.fill_parameters(stn, 5, gain=0.3)
    with torch.no_grad():
        stn.warp_head.linear.bias.copy_(torch.tensor([0.3, 0.2, 0.1, -0.1]))
        for mode in ("border", "reflection", "zeros"):
            out, grid, m = stn(blob["cfg1.x"], return_warp=True, return_flow=True, padding_mode=mode)
            assert_close(out, blob["cfg1.out." + mode], rtol=1e-4, what="config1 " + mode)
            assert_close(m, blob["cfg1.M"], rtol=1e-5)
            assert_close(grid, blob["cfg1.grid"], rtol=1e-5)


def test_state_dicts_are_key_compatible_with_the_reference():
    """The layouts (keys in order, shapes) of the reference's state dicts are kept in tests/golden/state_dicts.npz
    (conftest.Pinned)."""
    import importlib
    from gangealing_b200.stn import get_stn
    from gangealing_b200.training import DirectionInterpolator
    pin = Pinned("state_dicts")

    def ref(module):
        refimport.import_reference()
        torch.Tensor.cuda = lambda self, *a, **k: self  # reference FlowHead.__init__ calls .cuda() (warping_heads.py:158)
        return importlib.import_module(module)
    layout = pin.value("generator", lambda: state_dict_layout(ref("models.stylegan2.networks").Generator(32, 32, 2)))
    assert state_dict_layout(_gen()) == layout.tolist()
    for tr in (["similarity"], ["similarity", "flow"]):
        args = dict(flow_size=64, supersize=128, channel_multiplier=0.5, num_heads=2)
        layout = pin.value("stn." + "_".join(tr), lambda: state_dict_layout(
            ref("models.spatial_transformers.spatial_transformer").get_stn(list(tr), **args)))
        m = get_stn(list(tr), ops=CPU, **args)
        assert state_dict_layout(m) == layout.tolist()
        m.load_state_dict(zeros_state_dict(layout))
    layout = pin.value("latent_learner", lambda: state_dict_layout(ref("models.latent_learner").DirectionInterpolator(None, 3, 5, 14, num_heads=2)))
    assert state_dict_layout(DirectionInterpolator(None, 3, 5, 14, num_heads=2)) == layout.tolist()
    pin.save()


def test_train_step_runs_and_learns_on_cpu_oracle_ops():
    from gangealing_b200.training import TrainConfig, Trainer
    cfg = TrainConfig(gen_size=64, flow_size=64, dim_latent=32, n_mlp=2, batch=2, inject=3)
    tr = Trainer(cfg, "cpu", ops=CPU)
    before = [p.detach().clone() for p in tr.t_module.parameters()]
    ema_before = [p.detach().clone() for p in tr.t_ema.parameters()]
    out = tr.step()   # heads are zero-initialised: the first step only moves the heads' last layers ...
    out = tr.step()   # ... the second one reaches the trunks
    assert set(out) == {"p", "tv", "f"} and torch.isfinite(out["p"])
    changed = sum(int(not torch.equal(a, b)) for a, b in zip(before, tr.t_module.parameters()))
    assert changed > 10, "STN parameters did not move"
    assert any(not torch.equal(a, b) for a, b in zip(ema_before, tr.t_ema.parameters()))
    assert all(p.grad is None for p in tr.generator.parameters())  # G is frozen
    assert tr.ll_module.coefficients.grad is not None               # pass #2 of G is differentiated


@pytest.mark.parametrize("transforms", [("similarity",), ("similarity", "flow")])
def test_point_transfer_matches_reference_fixture(transforms):
    """congeal_points / uncongeal_points / transfer_points (reference spatial_transformer.py:631-720), SURVEY.md 8(a13):
    the nearest-neighbour indices of the flow STN (argmin + unravel_index) must match EXACTLY."""
    from gangealing_b200.stn import get_stn
    blob = load_golden("points")
    tag = "pts_" + "_".join(transforms)
    stn = get_stn(list(transforms), flow_size=64, supersize=64, channel_multiplier=0.25, num_heads=1, ops=CPU).eval()
    opset.fill_parameters(stn, 21, gain=0.3)
    img_a, img_b, pts = blob[tag + ".img_a"], blob[tag + ".img_b"], blob[tag + ".points"]
    with torch.no_grad():
        congealed = stn.congeal_points(img_a, pts)
        is_index = congealed.dtype != torch.float32
        back = stn.uncongeal_points(img_b, congealed.float() if is_index else congealed, normalize_input_points=is_index)
        moved = stn.transfer_points(img_a, img_b, pts)
    ref = blob[tag + ".congealed"]
    assert congealed.dtype == ref.dtype and congealed.shape == ref.shape
    if is_index:
        assert torch.equal(congealed, ref), "nearest-neighbour indices differ from the reference"
    else:
        assert_close(congealed, ref, rtol=1e-5, what="congealed points")
    assert_close(back, blob[tag + ".uncongealed"], rtol=1e-5, what="uncongealed points")
    assert_close(moved, blob[tag + ".transferred"], rtol=1e-5, what="transferred points")


def _flat(res):
    if torch.is_tensor(res):
        return [res]
    out = []
    for r in res:
        out += _flat(r)
    return out


def test_stn_orchestration_options_match_reference_fixture():
    """SURVEY.md 8(a11): iterated similarity, composed STN with alpha / output_resolution / return_sim /
    return_intermediates, multi-head cartesian policy and unfold -- same calls as oracle/make_golden.py made on the
    reference (spatial_transformer.py:78-139, :523-615)."""
    from gangealing_b200.stn import get_stn
    from oracle.make_golden import STN_OPTION_CASES, stn_option_kwargs
    blob = load_golden("stn_options")
    for i, (name, transforms, heads, kw) in enumerate(STN_OPTION_CASES):
        stn = get_stn(list(transforms), flow_size=64, supersize=64, channel_multiplier=0.25, num_heads=heads, ops=CPU).eval()
        opset.fill_parameters(stn, 31 + i, gain=0.3)
        with torch.no_grad():
            res = _flat(stn(blob["opt_" + name + ".x"], **stn_option_kwargs(kw)))
        expected = [blob[k] for k in sorted((k for k in blob if k.startswith("opt_" + name + ".out")),
                                            key=lambda k: int(k.rsplit("out", 1)[1]))]
        assert len(res) == len(expected), name
        for j, (a, e) in enumerate(zip(res, expected)):
            assert_close(a, e, rtol=2e-4, what="%s output %d" % (name, j))
