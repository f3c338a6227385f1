"""Per-image exposure, the parts that need no GPU: graphdeco's learning-rate schedule, the exposure table's bookkeeping
(mapping, exposure.json round trip) on CPU tensors, the trainer's refusal without a table, and the C-ABI's argument
checks (pointers are never dereferenced)."""
import math

import numpy as np
import pytest
import torch


def _lr_reference(step, lr_init, lr_final, delay_steps, delay_mult, max_steps):
    """graphdeco utils/general_utils.py get_expon_lr_func, written out with numpy."""
    if step < 0 or (lr_init == 0.0 and lr_final == 0.0):
        return 0.0
    delay = (delay_mult + (1 - delay_mult) * np.sin(0.5 * np.pi * np.clip(step / delay_steps, 0, 1))
             if delay_steps > 0 else 1.0)
    t = np.clip(step / max_steps, 0, 1)
    return float(delay * np.exp(np.log(lr_init) * (1 - t) + np.log(lr_final) * t))


def test_expon_lr_matches_graphdeco_schedule():
    from hidegs_b200.optim import get_expon_lr_func
    from hidegs_b200.trainer import OptimizationParams as O
    args = (O.exposure_lr_init, O.exposure_lr_final, O.exposure_lr_delay_steps, O.exposure_lr_delay_mult, O.iterations)
    f = get_expon_lr_func(*args[:4], max_steps=args[4])
    for step in (0, 1, 2500, 4999, 5000, 15_000, 29_999, 30_000, 45_000):
        assert f(step) == pytest.approx(_lr_reference(step, *args), rel=1e-12, abs=0.0), step
    # the values themselves: delay_mult * lr_init at 0, the sine ramp inside the delay, log-linear after, lr_final past
    # max_steps
    assert f(0) == pytest.approx(0.001 * 0.01, rel=1e-12)
    ramp = 0.001 + 0.999 * math.sin(0.25 * math.pi)
    assert f(2500) == pytest.approx(ramp * math.exp(math.log(0.01) * (1 - 2500 / 30000) + math.log(1e-4) * 2500 / 30000),
                                    rel=1e-12)
    assert f(15_000) == pytest.approx(math.sqrt(0.01 * 1e-4), rel=1e-12)
    assert f(45_000) == pytest.approx(1e-4, rel=1e-12)
    assert f(-1) == 0.0 and get_expon_lr_func(0.0, 0.0)(10) == 0.0
    g = get_expon_lr_func(0.02, 0.001, max_steps=100)  # no delay
    assert g(0) == pytest.approx(0.02, rel=1e-12) and g(100) == pytest.approx(0.001, rel=1e-12)


def _cpu_params(n=10):
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(0)
    return tr.GaussianParams(torch.randn(n, 3, generator=g), torch.randn(n, 16, 3, generator=g),
                             torch.randn(n, 1, generator=g), torch.randn(n, 3, generator=g) - 3,
                             torch.randn(n, 4, generator=g))


def test_exposure_table_bookkeeping_and_round_trip(tmp_path):
    from hidegs_b200 import ply_io
    p = _cpu_params()
    names = ["b.jpg", "a.jpg", "c.jpg"]
    p.setup_exposures(names)
    assert p.exposure_mapping == {"b.jpg": 0, "a.jpg": 1, "c.jpg": 2}
    assert p._exposure.shape == (3, 3, 4) and p._exposure.is_leaf and p._exposure.requires_grad
    assert torch.equal(p._exposure.detach(), torch.eye(3, 4).repeat(3, 1, 1))
    assert p._exposure.grad is p.exposure_grad and p.exposure_grad.data_ptr() != p._exposure.data_ptr()
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        p._exposure += 0.1 * torch.randn(3, 3, 4, generator=g)
    assert torch.equal(p.get_exposure_from_name("a.jpg").detach(), p._exposure[1].detach())
    path = str(tmp_path / "exposure.json")
    p.save_exposures(path)
    loaded = ply_io.load_exposures(path, device="cpu")
    assert list(loaded) == names  # mapping order
    q = _cpu_params()
    q.setup_exposures(names, exposures=loaded)
    assert torch.equal(q._exposure.detach(), p._exposure.detach())  # exact: json keeps the float32 values
    q2 = _cpu_params()
    q2.setup_exposures(list(reversed(names)), exposures=loaded)
    for n in names:
        assert torch.equal(q2.get_exposure_from_name(n).detach(), p.get_exposure_from_name(n).detach())
    with pytest.raises(ValueError):
        p.get_exposure_from_name("missing.jpg")
    with pytest.raises(ValueError):
        _cpu_params().setup_exposures(["x", "x"])
    with pytest.raises(ValueError):
        _cpu_params().setup_exposures(names + ["d.jpg"], exposures=loaded)
    with pytest.raises(ValueError):
        _cpu_params().get_exposure_from_name("a.jpg")  # no table


def test_train_exposure_needs_a_table():
    from hidegs_b200 import trainer as tr
    p = _cpu_params()
    with pytest.raises(ValueError, match="setup_exposures"):
        tr.ViewShardedTrainer(p, torch.zeros(3), train_exposure=True)
    tr.ViewShardedTrainer(p, torch.zeros(3))  # the default is off


def test_exposure_abi_rejects_bad_arguments():
    from hidegs_b200._losses_lib import lib
    L = lib()
    fake = 4096
    assert L.hg_exposure_apply(None, fake, 4, 4, fake, None) == 1
    assert b"hg_exposure_apply" in L.hg_last_error()
    assert L.hg_exposure_apply(fake, None, 4, 4, fake, None) == 1
    assert L.hg_exposure_apply(fake, fake, 4, 4, None, None) == 1
    assert L.hg_exposure_apply(fake, fake, 0, 4, fake, None) == 1
    assert L.hg_exposure_apply(fake, fake, 4, -1, fake, None) == 1
    assert L.hg_exposure_grad_workspace_bytes(0, 4) == 0
    assert L.hg_exposure_grad_workspace_bytes(1080, 1920) >= 12 * 8 * (1080 * 1920 // 1024)
    full = [fake, fake, fake, fake, fake, 4, 4, 0.8, -0.2, fake, fake, fake, fake, None]
    for i in (0, 1, 2, 10, 11, 12):  # color, exposure, gt, out, exposure_grad, workspace
        a = list(full)
        a[i] = None
        assert L.hg_training_image_grad_exposure(*a) == 1, i
        assert b"hg_training_image_grad_exposure" in L.hg_last_error()
    for i in (5, 6):
        for bad in (0, -3):
            a = list(full)
            a[i] = bad
            assert L.hg_training_image_grad_exposure(*a) == 1
