"""Monocular inverse-depth supervision, the parts that need no GPU: the weight schedule, depth_params.json, the camera-side
prior rules of graphdeco's Camera.__init__, the C-ABI's argument checks (pointers are never dereferenced) and the
trainer's refusal of a prior it cannot use."""
import json

import numpy as np
import pytest
import torch


def _expon_reference(step, init, final, max_steps):
    """graphdeco utils/general_utils.py get_expon_lr_func without a delay, written out with numpy."""
    if step < 0 or (init == 0.0 and final == 0.0):
        return 0.0
    t = np.clip(step / max_steps, 0, 1)
    return float(np.exp(np.log(init) * (1 - t) + np.log(final) * t))


def test_default_depth_weight_schedule():
    from hidegs_b200.optim import get_expon_lr_func
    from hidegs_b200.trainer import OptimizationParams as O
    assert (O.depth_l1_weight_init, O.depth_l1_weight_final) == (1.0, 0.01)
    f = get_expon_lr_func(O.depth_l1_weight_init, O.depth_l1_weight_final, max_steps=O.iterations)
    for step in (0, 1, 7, 1000, 15_000, 29_999, 30_000, 60_000):
        assert f(step) == pytest.approx(_expon_reference(step, 1.0, 0.01, O.iterations), rel=1e-12, abs=0.0), step
    assert f(0) == pytest.approx(1.0, rel=1e-12)
    assert f(15_000) == pytest.approx(0.1, rel=1e-12)
    assert f(30_000) == pytest.approx(0.01, rel=1e-12) and f(60_000) == pytest.approx(0.01, rel=1e-12)
    assert get_expon_lr_func(0.0, 0.0, max_steps=O.iterations)(10) == 0.0


def test_load_depth_params_median_of_positive_scales(tmp_path):
    from hidegs_b200 import ply_io
    path = tmp_path / "depth_params.json"
    path.write_text(json.dumps({"a": {"scale": 2.0, "offset": 0.1}, "b": {"scale": -1.0, "offset": 0.0},
                                "c": {"scale": 0.0, "offset": 0.3}, "d": {"scale": 4.0, "offset": -0.2},
                                "e": {"scale": 10.0, "offset": 0.0}}))
    p = ply_io.load_depth_params(str(path))
    assert set(p) == set("abcde")
    assert all(v["med_scale"] == 4.0 for v in p.values())  # median of 2, 4, 10: the non-positive ones do not count
    assert p["a"]["scale"] == 2.0 and p["d"]["offset"] == -0.2
    path.write_text(json.dumps({"a": {"scale": 0.0, "offset": 0.1}, "b": {"scale": -2.0, "offset": 0.0}}))
    assert all(v["med_scale"] == 0.0 for v in ply_io.load_depth_params(str(path)).values())


class _Cam:
    image_height, image_width, image_name = 3, 4, "cam"


def _map():
    return torch.tensor([[-0.5, 0.0, 0.25, 1.0], [2.0, -3.0, 0.5, 0.75], [0.1, 0.2, -0.01, 4.0]], dtype=torch.float32)


def test_attach_depth_prior_rules():
    from hidegs_b200.ply_io import attach_depth_prior
    inv = _map()
    clamped = inv.clamp_min(0)
    # no depth_params: clamped, reliable, mask kept as given (None = all ones)
    cam = attach_depth_prior(_Cam(), inv)
    assert cam.depth_reliable and cam.depth_mask is None
    assert cam.invdepthmap.shape == (1, 3, 4) and cam.invdepthmap.dtype == torch.float32
    assert torch.equal(cam.invdepthmap[0], clamped)
    assert torch.equal(inv, _map())  # the caller's map is not modified
    # the clamp comes BEFORE scale and offset: a negative value becomes `offset`, not `scale * v + offset` clamped
    dp = dict(scale=2.0, offset=-0.25, med_scale=2.0)
    cam = attach_depth_prior(_Cam(), inv.numpy(), dp)
    assert cam.depth_reliable
    assert torch.equal(cam.invdepthmap[0], clamped * 2.0 + (-0.25))
    assert float(cam.invdepthmap[0, 0, 0]) == -0.25 and float(cam.invdepthmap[0, 1, 1]) == -0.25
    # reliability bounds: scale < 0.2 med or scale > 5 med is unreliable (mask zeroed); both sides of each bound
    mask = torch.full((1, 3, 4), 0.5)
    for scale, reliable in ((0.39, False), (0.4, True), (0.41, True), (9.9, True), (10.0, True), (10.1, False)):
        cam = attach_depth_prior(_Cam(), inv, dict(scale=scale, offset=0.0, med_scale=2.0), mask=mask)
        assert cam.depth_reliable == reliable, scale
        assert torch.equal(cam.depth_mask, mask if reliable else torch.zeros_like(mask)), scale
        assert torch.equal(cam.invdepthmap[0], clamped * scale), scale  # (scaled either way: scale > 0)
    cam = attach_depth_prior(_Cam(), inv, dict(scale=100.0, offset=0.0, med_scale=2.0))
    assert not cam.depth_reliable and torch.equal(cam.depth_mask, torch.zeros(1, 3, 4))
    # scale <= 0 leaves the map unscaled (and without its offset); with med_scale 0 a zero scale is still reliable
    for scale in (0.0, -1.5):
        cam = attach_depth_prior(_Cam(), inv, dict(scale=scale, offset=0.7, med_scale=0.0))
        assert torch.equal(cam.invdepthmap[0], clamped), scale
        assert cam.depth_reliable == (scale == 0.0), scale
    # shapes: [H, W] and [1, H, W] are both taken; anything else raises
    attach_depth_prior(_Cam(), inv[None])
    for bad in (inv.t(), inv[:, :3], inv[None, None], torch.zeros(2, 3, 4)):
        with pytest.raises(ValueError, match="shape"):
            attach_depth_prior(_Cam(), bad)
    with pytest.raises(ValueError, match="mask"):
        attach_depth_prior(_Cam(), inv, mask=torch.ones(4, 3))


def test_invdepth_l1_abi_rejects_bad_arguments():
    from hidegs_b200._losses_lib import lib
    L = lib()
    fake = 4096
    assert L.hg_invdepth_l1_workspace_bytes(0, 4) == 0 and L.hg_invdepth_l1_workspace_bytes(4, -1) == 0
    assert L.hg_invdepth_l1_workspace_bytes(1080, 1920) >= 8 * (1080 * 1920 // 4096)
    full = [fake, fake, fake, 4, 4, 1.0, fake, fake, fake, fake, None]
    for i in (0, 1, 6, 7, 9):  # invdepth, mono, grad, value, workspace
        a = list(full)
        a[i] = None
        assert L.hg_invdepth_l1(*a) == 1, i
        assert b"hg_invdepth_l1" in L.hg_last_error()
    for i in (3, 4):
        for bad in (0, -2):
            a = list(full)
            a[i] = bad
            assert L.hg_invdepth_l1(*a) == 1, (i, bad)


def _cpu_params(n=10):
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(0)
    return tr.GaussianParams(torch.randn(n, 3, generator=g), torch.randn(n, 16, 3, generator=g),
                             torch.randn(n, 1, generator=g), torch.randn(n, 3, generator=g) - 3,
                             torch.randn(n, 4, generator=g))


def test_trainer_refuses_unusable_priors_before_the_step():
    from hidegs_b200 import trainer as tr
    from hidegs_b200.ply_io import attach_depth_prior
    p = _cpu_params()
    trainer = tr.ViewShardedTrainer(p, torch.zeros(3), depth_regularization=True)
    arena = p.param_arena.clone()
    gt = torch.zeros(3, 3, 4)
    bad = []
    bad.append(attach_depth_prior(_Cam(), torch.ones(3, 4), device="meta"))           # another device
    c = attach_depth_prior(_Cam(), torch.ones(3, 4))
    c.depth_mask = torch.ones(1, 3, 4, device="meta")                                  # mask on another device
    bad.append(c)
    c = _Cam()
    c.invdepthmap, c.depth_reliable = torch.ones(1, 4, 3), True                        # wrong shape
    bad.append(c)
    c = attach_depth_prior(_Cam(), torch.ones(3, 4))
    c.depth_mask = torch.ones(3, 4)                                                    # mask without its channel
    bad.append(c)
    c = attach_depth_prior(_Cam(), torch.ones(3, 4))
    c.invdepthmap = c.invdepthmap.double()                                             # not float32
    bad.append(c)
    for cam in bad:
        with pytest.raises(ValueError):
            trainer.step([(cam, gt)])
        assert trainer.iteration == 0 and torch.equal(p.param_arena, arena)
    # an unreliable prior is not looked at: it takes no part in the loss
    c = _Cam()
    c.invdepthmap, c.depth_reliable = torch.ones(1, 4, 3), False
    assert trainer._depth_prior(c) is None and trainer._depth_prior(_Cam()) is None
    # off by default: the same cameras are not looked at either
    assert tr.ViewShardedTrainer(p, torch.zeros(3))._depth_term(bad[0], 1) is None
