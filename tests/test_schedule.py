"""psi annealing / cyclic learning rate (training/schedule.py) against the reference's utils/annealing.py, and the
Trainer's device-resident psi / lr scalars (the captured step reads them at replay time)."""
import math

import pytest
import torch

from conftest import Pinned
from gangealing_b200.training import schedule as S
from oracle import refimport


def test_closed_forms():
    assert S.psi_at(0, 100)[0] == pytest.approx(1.0) and S.psi_at(100, 100) == (pytest.approx(0.0, abs=1e-12), False)
    assert S.psi_at(101, 100) == (0.0, True)
    assert S.psi_at(50, 100, "linear")[0] == pytest.approx(0.5) and S.psi_at(50, 100, "cosine")[0] == pytest.approx(0.5)
    # T_0 = 1, T_mult = 2: restarts at epochs 1, 3, 7, ... each cycle's peak decayed by 0.9
    assert S.decaying_cosine_lr(0.0, 1e-3) == pytest.approx(1e-3)
    assert S.decaying_cosine_lr(0.5, 1e-3) == pytest.approx(0.5e-3)
    assert S.decaying_cosine_lr(1.0, 1e-3) == pytest.approx(0.9e-3)
    assert S.decaying_cosine_lr(2.0, 1e-3) == pytest.approx(0.45e-3)
    assert S.decaying_cosine_lr(3.0, 1e-3) == pytest.approx(0.81e-3)
    assert S.lr_cycle_iters(150000, 37500, 1500000, 2) == [149999, 187499, 262499, 412499, 712499, 1312499]
    s = S.schedule_at(150000 + 37500 // 2, 1e-3, 1e-2)
    assert s["psi"] == 0.0 and s["stn_lr"] == pytest.approx(0.5e-3) and s["ll_lr"] == pytest.approx(0.5e-2)


def test_against_the_reference_scheduler_and_annealers():
    """What the reference's utils/annealing.py computes is kept in tests/golden/schedule.npz (conftest.Pinned)."""
    pin = Pinned("schedule")

    def annealing():
        import importlib.util
        import os
        spec = importlib.util.spec_from_file_location("ref_annealing", os.path.join(refimport.REFERENCE_ROOT, "utils", "annealing.py"))
        A = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(A)
        return A
    for fn in ("cosine", "linear"):
        for i in (0, 1, 777, 149999, 150000):
            want = pin.value("psi.%s.%d" % (fn, i), lambda: float(annealing().get_psi_annealing_fn(fn)(i, 1.0, 0.0, 150000)))
            assert S.psi_at(i, 150000, fn)[0] == pytest.approx(float(want), abs=1e-6)
    want = pin.value("lr_cycle_iters", lambda: annealing().lr_cycle_iters(150000, 37500, 1500000, 2))
    assert S.lr_cycle_iters(150000, 37500, 1500000, 2) == want.tolist()
    epochs = [0.0, 0.01, 0.5, 0.999, 1.0, 1.7, 2.99, 3.0, 6.5, 7.0, 12.345, 31.0]

    def reference_lrs():
        net = torch.nn.Linear(2, 2)
        opt = torch.optim.SGD(net.parameters(), 1e-3)
        sched = annealing().DecayingCosineAnnealingWarmRestarts(opt, T_0=1, T_mult=2, decay=0.9)
        lrs = []
        for epoch in epochs:
            sched.step(epoch)
            lrs.append(opt.param_groups[0]["lr"])
        return lrs
    for epoch, lr in zip(epochs, pin.value("decaying_cosine_lr", reference_lrs).tolist(), strict=True):
        assert S.decaying_cosine_lr(epoch, 1e-3, 2, 0.9) == pytest.approx(lr, rel=1e-9, abs=1e-15), epoch
    pin.save()


def test_trainer_schedule_scalars_on_cpu():
    from gangealing_b200.training import TrainConfig, Trainer
    from oracle import opset
    cfg = TrainConfig(gen_size=64, flow_size=64, dim_latent=32, n_mlp=2, batch=1, inject=3, stn_channel_multiplier=0.125,
                      gen_channel_multiplier=1)
    tr = Trainer(cfg, "cpu", ops=opset.cpu_ops())
    s = tr.set_iteration(10, anneal_psi=20, period=10.0)
    assert float(tr.psi_t) == pytest.approx(0.5) and s["stn_lr"] == cfg.stn_lr
    s = tr.set_iteration(25, anneal_psi=20, period=10.0)
    assert float(tr.psi_t) == 0.0
    assert tr.t_optim.param_groups[0]["lr"] == pytest.approx(0.5 * cfg.stn_lr)
    assert tr.ll_optim.param_groups[0]["lr"] == pytest.approx(0.5 * cfg.ll_lr)
    # psi reaches the latent learner as a tensor: psi = 1 leaves the sampled latent untouched (no truncation)
    w = torch.randn(2, cfg.dim_latent)
    tr.set_schedule(psi=1.0)
    out = tr.ll([w], psi=tr.psi_t)[0]
    assert torch.allclose(out[:, 0], w, atol=1e-6)
    tr.step(psi=0.3, lr=1e-4, ll_lr=2e-4)
    assert float(tr.psi_t) == pytest.approx(0.3) and tr.t_optim.param_groups[0]["lr"] == pytest.approx(1e-4)
    assert math.isfinite(float(tr.step()["p"]))
