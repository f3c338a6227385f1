"""Camera pose refinement, the parts that need no GPU: the host SO(3) helpers against scipy, the pose table's
bookkeeping and camera_poses.json round trip on CPU tensors, the trainer's refusals, and the C-ABI's argument checks
(pointers are never dereferenced)."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

from hidegs_b200 import camera_pose as cp

PHIS = ([0.0, 0.0, 0.0], [1e-9, -2e-9, 3e-9], [3e-5, -1e-5, 2e-5], [0.3, -0.2, 0.1], [1.2, 0.4, -2.0],
        [0.0, 3.0, 0.0])


@pytest.mark.parametrize("phi", PHIS)
def test_so3_exp_matches_scipy(phi):
    R = cp.so3_exp(phi)
    assert np.allclose(R, Rotation.from_rotvec(phi).as_matrix(), rtol=0, atol=1e-14)


@pytest.mark.parametrize("phi", PHIS)
def test_left_jacobian_matches_scipy_differences(phi):
    """Exp(phi + d) Exp(phi)^T = Exp(J_l(phi) d) to first order: central differences of scipy's log map."""
    phi = np.asarray(phi, dtype=np.float64)
    J = cp.so3_left_jacobian(phi)
    R0 = Rotation.from_rotvec(phi)
    h = 1e-6
    num = np.zeros((3, 3))
    for k in range(3):
        d = np.zeros(3)
        d[k] = h
        plus = (Rotation.from_rotvec(phi + d) * R0.inv()).as_rotvec()
        minus = (Rotation.from_rotvec(phi - d) * R0.inv()).as_rotvec()
        num[:, k] = (plus - minus) / (2 * h)
    assert np.allclose(J, num, rtol=0, atol=1e-8)
    if not phi.any():
        assert np.array_equal(J, np.eye(3))


def test_pose_matrix_and_corrected_w2c():
    xi = np.array([0.1, -0.2, 0.3, 0.05, -0.02, 0.01])
    C = cp.pose_matrix(xi)
    assert np.allclose(C[:3, :3], Rotation.from_rotvec(xi[3:]).as_matrix(), atol=1e-14)
    assert np.array_equal(C[:3, 3], xi[:3]) and np.array_equal(C[3], [0, 0, 0, 1])
    from hidegs_b200 import synthetic as syn
    cam = syn.default_camera(64, 48, eye=(0.3, 0.1, -5.0))
    V = cam.world_view_transform.double().numpy()
    W2C = cp.corrected_w2c(V, xi)
    p = np.array([0.2, -0.4, 1.5, 1.0])
    # p_cam' = Exp(phi) p_cam + rho
    p_cam = (p @ V)[:3]
    assert np.allclose(W2C @ p, np.r_[cp.so3_exp(xi[3:]) @ p_cam + xi[:3], 1.0], atol=1e-12)
    assert np.array_equal(cp.corrected_w2c(V, np.zeros(6)), V.T)


def _cpu_params(n=10):
    from hidegs_b200 import trainer as tr
    g = torch.Generator().manual_seed(0)
    return tr.GaussianParams(torch.randn(n, 3, generator=g), torch.randn(n, 16, 3, generator=g),
                             torch.randn(n, 1, generator=g), torch.randn(n, 3, generator=g) - 3,
                             torch.randn(n, 4, generator=g))


def test_pose_table_bookkeeping_and_round_trip(tmp_path):
    from hidegs_b200 import ply_io, synthetic as syn
    p = _cpu_params()
    names = ["b.jpg", "a.jpg", "c.jpg"]
    p.setup_camera_poses(names)
    assert p.camera_pose_mapping == {"b.jpg": 0, "a.jpg": 1, "c.jpg": 2}
    assert p._camera_pose.shape == (3, 8) and p._camera_pose.is_leaf and p._camera_pose.requires_grad
    assert not p._camera_pose.detach().any()
    assert p._camera_pose.grad is p.camera_pose_grad and p.camera_pose_grad.data_ptr() != p._camera_pose.data_ptr()
    assert p.camera_pose_index("c.jpg") == 2
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        p._camera_pose[:, :6] += 0.01 * torch.randn(3, 6, generator=g)
    cams = []
    for k, n in enumerate(names[:2]):
        c = syn.default_camera(64, 48, eye=(0.2 * k, 0.0, -5.0))
        c.image_name = n
        cams.append(c)
    path = str(tmp_path / "camera_poses.json")
    p.save_camera_poses(path, cams)
    import json
    raw = json.load(open(path))
    assert list(raw) == names and "w2c" in raw["b.jpg"] and "w2c" in raw["a.jpg"] and "w2c" not in raw["c.jpg"]
    xi_a = p._camera_pose.detach()[1, :6].double().numpy()
    assert np.allclose(np.array(raw["a.jpg"]["w2c"]),
                       cp.corrected_w2c(cams[1].world_view_transform.double().numpy(), xi_a), atol=1e-12)
    loaded = ply_io.load_camera_poses(path)
    q = _cpu_params()
    q.setup_camera_poses(list(reversed(names)), poses=loaded)
    for n in names:  # exact: json keeps the float32 values
        assert torch.equal(q._camera_pose[q.camera_pose_index(n)].detach(), p._camera_pose[p.camera_pose_index(n)].detach())
    with pytest.raises(ValueError):
        p.camera_pose_index("missing.jpg")
    with pytest.raises(ValueError):
        _cpu_params().setup_camera_poses(["x", "x"])
    with pytest.raises(ValueError):
        _cpu_params().setup_camera_poses(names + ["d.jpg"], poses=loaded)
    with pytest.raises(ValueError):
        _cpu_params().setup_camera_poses(["x"], poses={"x": [0.0] * 5})
    with pytest.raises(ValueError):
        _cpu_params().camera_pose_index("a.jpg")  # no table


def test_train_poses_refusals(monkeypatch):
    from hidegs_b200 import trainer as tr
    p = _cpu_params()
    with pytest.raises(ValueError, match="setup_camera_poses"):
        tr.ViewShardedTrainer(p, torch.zeros(3), train_poses=True)
    p.setup_camera_poses(["a"])
    with pytest.raises(ValueError, match="CUDA"):
        tr.ViewShardedTrainer(p, torch.zeros(3), train_poses=True)
    monkeypatch.setenv("HG_TRAINER_DIRECT", "0")
    p.fused = True  # (pretend: the refusal of the autograd path comes before any device work)
    with pytest.raises(ValueError, match="HG_TRAINER_DIRECT"):
        tr.ViewShardedTrainer(p, torch.zeros(3), train_poses=True)
    p.fused = False
    with pytest.raises(ValueError, match="CUDA"):
        p.corrected_camera(type("Cam", (), {"image_name": "a"})())
    monkeypatch.delenv("HG_TRAINER_DIRECT")
    t = tr.ViewShardedTrainer(_cpu_params(), torch.zeros(3))  # the default is off
    assert not t.train_poses


def test_camera_pose_abi_rejects_bad_arguments():
    from hidegs_b200 import _lib
    from hidegs_b200._geometry_lib import lib
    L = lib()
    fake = 1 << 20  # never dereferenced: every call below fails its argument check first
    assert L.hg_camera_pose_apply(fake, fake, fake, fake, 3, 3, fake, None) == 1
    assert b"index 3" in L.hg_last_error()
    assert L.hg_camera_pose_apply(fake, fake, fake, fake, 3, -1, fake, None) == 1
    assert L.hg_camera_pose_apply(None, fake, fake, fake, 3, 0, fake, None) == 1
    assert L.hg_camera_pose_apply(fake, fake, fake, fake, 0, 0, fake, None) == 1
    assert L.hg_camera_pose_workspace_bytes(0) == 0 and L.hg_camera_pose_workspace_bytes(-5) == 0
    assert L.hg_camera_pose_workspace_bytes(1 << 31) == 0
    # [ceil(N / 128) rows | ceil(N / 256) rows] of 8 doubles, each part 256-byte aligned
    up = lambda b: (b + 255) // 256 * 256  # noqa: E731
    assert L.hg_camera_pose_workspace_bytes(1000) == up(8 * 64) + up(4 * 64)
    assert L.hg_camera_pose_workspace_bytes(2_000_000) == up(15625 * 64) + up(7813 * 64)
    assert L.hg_camera_pose_grad_finish(fake, 3, 3, 100, fake, fake, None, None) == 1
    assert L.hg_camera_pose_grad_finish(fake, 3, 0, 0, fake, fake, None, None) == 1
    assert L.hg_camera_pose_grad_finish(fake, 3, 0, 100, fake + 4, fake, None, None) == 1
    assert L.hg_camera_pose_grad_finish(None, 3, 0, 100, fake, fake, None, None) == 1
    args = [fake] * 4 + [100, 48, fake, fake, fake] + [None] * 8 + [0.0] + [fake] * 5
    assert L.hg_prologue_backward_pose(*args, None, None) == 1
    assert b"pose_workspace is NULL" in L.hg_last_error()
    assert L.hg_prologue_backward_pose(*args, fake + 8, None) == 1
    assert b"16-byte" in L.hg_last_error()
    # the rasterizer's pose backward: NULL workspace, render indices
    R = _lib.lib()
    ins = _lib.RasterInputs(P=100, N=100, D=0, M=1, W=16, H=16, tan_fovx=0.5, tan_fovy=0.5, scale_modifier=1.0,
                            background=fake, viewmatrix=fake, projmatrix=fake, campos=fake, means3D=fake, shs=fake,
                            opacities=fake, scales=fake, rotations=fake)
    cb = _lib.CHUNK_FN(0)
    ptrs = [fake] * 21
    assert R.hg_raster_backward_pose(ctypes.byref(ins), 0, *ptrs, 1, cb, None, None, 0.0, None, 0, None, None) == 1
    assert b"pose_workspace is NULL" in R.hg_last_error()
    ins.indices = fake
    assert R.hg_raster_backward_pose(ctypes.byref(ins), 0, *ptrs, 1, cb, None, None, 0.0, None, 0, fake, None) == 1
    assert b"render or parent indices" in R.hg_last_error()
    ins.indices = None
    ins.P = 50
    assert R.hg_raster_backward_pose(ctypes.byref(ins), 0, *ptrs, 1, cb, None, None, 0.0, None, 0, fake, None) == 1
