"""CPU: the cluster classifier (BASELINE config 5, second half) -- this repo's ResnetClassifier mirror and the
train_cluster_classifier.py iteration on the oracle op set against the fixture the REFERENCE produced
(oracle/make_golden.py:gen_classifier): logits, exact index outputs of the run_* helpers, `accuracy`, one training step."""
import pytest
import torch
from torch import nn, optim

from conftest import Pinned, assert_close, load_golden, state_dict_layout, zeros_state_dict
from oracle import opset, refimport
from oracle.make_golden import classifier_decimate, classifier_setup

CPU = opset.cpu_ops()


def _mods():
    from gangealing_b200.cluster_classifier import ResnetClassifier
    from gangealing_b200.stn import BilinearDownsample, get_stn
    from gangealing_b200.stylegan2 import Generator
    from gangealing_b200.training import DirectionInterpolator

    def with_ops(cls):
        return lambda *a, **k: cls(*a, ops=CPU, **k)
    return dict(Generator=with_ops(Generator), get_stn=with_ops(get_stn), DirectionInterpolator=DirectionInterpolator,
                ResnetClassifier=with_ops(ResnetClassifier), BilinearDownsample=with_ops(BilinearDownsample))


def _mse(a, b):
    return (a - b).pow(2).mean(dim=(1, 2, 3))


def test_classifier_forward_and_inference_helpers_match_reference_fixture():
    blob = load_golden("classifier")
    _, _, _, cls, _, clusters = classifier_setup(_mods())
    x = blob["cls.x"]
    with torch.no_grad():
        assert_close(cls(x), blob["cls.logits"], rtol=1e-4, what="logits")
        assert torch.equal(cls.assign(x), blob["cls.assign"])
        assert torch.equal(cls.assign(x, ignore_flips=True), blob["cls.assign_noflip"])
        for c in range(clusters // 2):
            kept, preds, flip, keep = cls.run(x, c, return_flip_indices=True)
            assert torch.equal(keep, blob["cls.run%d.keep" % c]) and torch.equal(flip, blob["cls.run%d.flip" % c])
            assert torch.equal(classifier_decimate(kept), blob["cls.run%d.kept" % c])       # a selection + mirror: exact
            assert_close(preds, blob["cls.run%d.preds" % c], rtol=1e-4)
            two = cls.run(x, c)
            assert len(two) == 2 and torch.equal(two[0], kept)
            flipped, flip_t = cls.run_flip_target(x, c)
            assert torch.equal(flip_t, blob["cls.run_flip_target%d.flip" % c])
            assert torch.equal(classifier_decimate(flipped), blob["cls.run_flip_target%d.out" % c])
        flipped, preds, classes, flip = cls.run_flip(x)
        assert torch.equal(classes, blob["cls.run_flip.classes"]) and torch.equal(flip, blob["cls.run_flip.flip"])
        assert torch.equal(classifier_decimate(flipped), blob["cls.run_flip.out"])
        tiled, policy = cls.run_flip_cartesian(x)
        assert torch.equal(policy, blob["cls.cartesian.policy"])
        assert torch.equal(classifier_decimate(tiled), blob["cls.cartesian.out"])


def test_reverse_topk_accuracy_matches_reference_fixture():
    from gangealing_b200.cluster_classifier import accuracy
    blob = load_golden("classifier")
    for k in (1, 2, 3):
        assert accuracy(blob["acc.pred"], blob["acc.gt"], k=k).item() == blob["acc.k%d" % k].item()


def test_classifier_training_iteration_matches_reference_fixture():
    """train_cluster_classifier.py:84-105 -- assignments by the frozen clustering STN (exact), cross-entropy, accuracies,
    head histograms, classifier gradients and the parameters after one Adam step."""
    from gangealing_b200.cluster_classifier import accuracy
    from gangealing_b200.training import assign_fake_images_to_clusters
    blob = load_golden("classifier")
    g, stn, ll, cls, resize, clusters = classifier_setup(_mods())
    batch = 3
    cls_optim = optim.Adam(cls.parameters(), lr=0.001)
    torch.manual_seed(4321)
    with torch.no_grad():
        assigned, _, _, _, resized, distance = assign_fake_images_to_clusters(
            g, stn, ll, _mse, resize, 0.0, batch, 512, True, 2, True, "cpu", sample_from_full_res=True, z=None,
            padding_mode="reflection")
    assert torch.equal(assigned.indices, blob["step.assignments"])
    assert_close(distance, blob["step.distance"], rtol=2e-4, what="cluster distances")
    logits = cls(resized[:batch])
    loss = nn.CrossEntropyLoss()(logits, assigned.indices)
    assert_close(logits, blob["step.logits"], rtol=2e-4, what="logits")
    assert_close(loss, blob["step.xent"], rtol=1e-4, what="cross entropy")
    assert accuracy(logits, -distance).item() == blob["step.acc1"].item()
    assert accuracy(logits, -distance, k=2).item() == blob["step.acc2"].item()
    cls.zero_grad()
    loss.backward()
    params = dict(cls.named_parameters())
    grads = [k for k in blob if k.startswith("step.grad.")]
    assert len(grads) >= 4
    for k in grads:
        assert_close(params[k[len("step.grad."):]].grad, blob[k], rtol=2e-3, what=k)
    cls_optim.step()
    assert_close(cls.to_logits.bias, blob["step.after.to_logits.bias"], rtol=1e-4)
    assert_close(cls.final_conv[1].bias, blob["step.after.final_conv.1.bias"], rtol=1e-4)


def test_classifier_trainer_step_reports_the_reference_loss_dict_and_learns():
    """ClassifierTrainer (training/classifier_step.py) on the oracle op set: keys of the reference's loss dict, head histograms
    that sum to one, a classifier initialised from the similarity STN's trunk, parameters that move, frozen everything else."""
    from gangealing_b200.training import TrainConfig, Trainer
    from gangealing_b200.training.classifier_step import ClassifierTrainer
    cfg = TrainConfig(gen_size=128, flow_size=64, dim_latent=32, n_mlp=2, batch=3, inject=3, num_heads=2, flips=True, ndirs=2,
                      sample_from_full_res=True, padding_mode="reflection", stn_channel_multiplier=0.25, gen_channel_multiplier=1)
    tr = Trainer(cfg, "cpu", ops=CPU)
    ct = ClassifierTrainer(tr, cls_lr=1e-3, ops=CPU)
    trunk = dict(tr.t_ema.stns[0].named_parameters())
    for name, p in ct.module.named_parameters():
        if name.startswith(("convs.", "final_conv.")):
            assert torch.equal(p, trunk[name]), "classifier trunk is not the similarity STN's (%s)" % name
    before = [p.detach().clone() for p in ct.module.parameters()]
    stn_before = [p.detach().clone() for p in tr.t_ema.parameters()]
    out = ct.step()
    assert set(out) == {"cross_entropy", "acc@1", "acc@2"} | {"head_%d" % c for c in range(4)} | {"pred_head_%d" % c for c in range(4)}
    assert torch.isfinite(out["cross_entropy"])
    assert abs(sum(float(out["head_%d" % c]) for c in range(4)) - 1.0) < 1e-6
    assert abs(sum(float(out["pred_head_%d" % c]) for c in range(4)) - 1.0) < 1e-6
    assert sum(int(not torch.equal(a, b)) for a, b in zip(before, ct.module.parameters())) > 10
    assert all(torch.equal(a, b) for a, b in zip(stn_before, tr.t_ema.parameters()))
    assert all(p.grad is None for p in tr.generator.parameters())
    lr0 = ct.set_iteration(0)
    assert lr0 == pytest.approx(1e-3) and ct.set_iteration(37500 // 2) == pytest.approx(0.5e-3)


def test_classifier_state_dict_is_key_compatible_with_the_reference():
    """The layout (keys in order, shapes) of the reference classifier's state dict is kept in
    tests/golden/state_dicts_classifier.npz (conftest.Pinned)."""
    from gangealing_b200.cluster_classifier import ResnetClassifier
    pin = Pinned("state_dicts_classifier")

    def reference():
        refimport.import_reference()
        from models import ResnetClassifier as Ref
        return state_dict_layout(Ref(64, channel_multiplier=0.5, num_heads=8, supersize=256))
    layout = pin.value("resnet_classifier", reference)
    m = ResnetClassifier(64, channel_multiplier=0.5, num_heads=8, supersize=256, ops=CPU)
    assert state_dict_layout(m) == layout.tolist()
    m.load_state_dict(zeros_state_dict(layout))
    pin.save()
