"""GPU parity tests of the rasterizer hot path (run on the B200 box: `pytest -m gpu`).

Every test calls the product path through the C-ABI (hidegs_b200._C -> ctypes ->
libhidegs_b200.so) and compares with
  * the UNMODIFIED reference CUDA rasterizer built for sm_100 (oracle/_ref, when present),
  * golden fixtures produced by that reference (tests/golden/raster_ref_*.npz),
  * the CPU restatement (oracle/raster_oracle.c) on small seeded scenes,
and, at BASELINE.json's full size, through size-independent properties.

Tolerances (BASELINE.json north_star): tile keys / sort order / tile ranges bit-exact;
images and depths <= 1e-4 absolute; gradients <= 1e-3 relative.
"""
import glob
import json
import os

import numpy as np
import pytest
import torch

import raster_utils as ru
from hidegs_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-4
CASES = {
    "plain": dict(n=6000, W=208, H=120, seed=21),
    "hier": dict(n=6000, W=208, H=120, seed=22, with_hier=True),
    "raw_indices": dict(n=6000, W=208, H=120, seed=23, with_hier=True, with_indices=True),
    "raw_indices_d0": dict(n=6000, W=208, H=120, seed=25, with_hier=True, with_indices=True, sh_degree=0),
    "ragged": dict(n=4000, W=203, H=117, seed=24),
}


def run_ours(case, dev, render_geo=True, do_depth=True, colors_precomp=None, backward=True):
    fa = ru.op_args(case, dev, render_geo=render_geo, do_depth=do_depth, colors_precomp=colors_precomp)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    grads = syn.upstream_grads(case["W"], case["H"], do_depth=do_depth)
    bwd = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, fwd, grads, dev)) if backward else None
    torch.cuda.synchronize()
    return fa, fwd, grads, bwd


def img_close(a, b, atol=IMG_ATOL, rtol=0.0, max_outliers=0):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    bad = (a - b).abs() > atol + rtol * b.abs()
    return int(bad.sum()) <= max_outliers


# ------------------------------------------------------------------ vs reference (GPU)
@pytest.mark.parametrize("name", list(CASES))
def test_bit_exact_binning_and_images_vs_reference(cuda_device, name):
    if not ru.ref_available():
        pytest.skip("oracle/_ref/ref_rasterizer_C.so not built")
    dev = cuda_device
    p = CASES[name]
    case = ru.build_case(**p)
    fa, ours, grads, ours_b = run_ours(case, dev)
    REF = ru.ref_module()
    ref = REF.rasterize_gaussians(*fa)
    ref_b = REF.rasterize_gaussians_backward(*ru.bwd_args(fa, ref, grads, dev))
    torch.cuda.synchronize()
    so, sr = ru.our_state(ours, case["P"], p["W"], p["H"]), ru.ref_state(ref, case["P"], p["W"], p["H"])
    assert ours[0] == ref[0] and ours[0] > 0
    for k in ("keys_unsorted", "keys", "point_list", "ranges", "n_contrib", "tiles_touched"):
        assert torch.equal(so[k], sr[k]), k
    assert torch.equal(ours[2], ref[2])  # radii
    assert torch.equal(ours[3], ref[3])  # out_observe
    assert torch.equal(so["final_T"].view(torch.int32), sr["final_T"].view(torch.int32))
    for i in (1, 4, 9):  # color, all_map, invdepth
        assert img_close(ours[i], ref[i]), i
    assert img_close(ours[5], ref[5], atol=IMG_ATOL, rtol=1e-5)  # plane depth is a quotient
    a = ru.mask_undefined_parent_rows(case, dict(zip(ru.GRAD_NAMES, ours_b)))
    b = ru.mask_undefined_parent_rows(case, dict(zip(ru.GRAD_NAMES, ref_b)))
    ru.assert_grads_close([a[n] for n in ru.GRAD_NAMES], [b[n] for n in ru.GRAD_NAMES], what=name)


# ------------------------------------------------------------------ vs golden fixtures
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "raster_ref_*.npz"))))
def test_against_reference_golden(cuda_device, path):
    dev = cuda_device
    gold = np.load(path)
    p = json.loads(bytes(gold["params"]).decode())
    case = ru.build_case(p["n"], p["W"], p["H"], seed=p["seed"], with_hier=p["with_hier"], with_indices=p["with_indices"],
                         sh_degree=p.get("sh_degree", 3))
    fa, ours, grads, ours_b = run_ours(case, dev, render_geo=p["render_geo"], do_depth=p["do_depth"])
    so = ru.our_state(ours, case["P"], p["W"], p["H"])
    assert ours[0] == int(gold["num_rendered"])
    assert np.array_equal(ours[2].cpu().numpy(), gold["radii"])
    if ours[0] > 0:
        for k in ("keys", "point_list", "keys_unsorted"):
            assert np.array_equal(so[k].cpu().numpy(), gold[k]), k
    for k in ("ranges", "n_contrib", "tiles_touched"):
        assert np.array_equal(so[k].cpu().numpy(), gold[k]), k
    assert np.array_equal(ours[3].cpu().numpy(), gold["out_observe"])
    assert img_close(ours[1], gold["color"]) and img_close(ours[4], gold["all_map"])
    assert img_close(ours[5], gold["plane_depth"], rtol=1e-5) and img_close(ours[9], gold["invdepth"])
    a = ru.mask_undefined_parent_rows(case, dict(zip(ru.GRAD_NAMES, ours_b)))
    b = ru.mask_undefined_parent_rows(case, {n: torch.from_numpy(gold[n]) for n in ru.GRAD_NAMES})
    ru.assert_grads_close([a[n] for n in ru.GRAD_NAMES], [b[n] for n in ru.GRAD_NAMES], what=os.path.basename(path))


# ------------------------------------------------------------------ vs CPU oracle
@pytest.mark.parametrize("name", list(CASES))
def test_parity_vs_cpu_oracle(cuda_device, name):
    dev = cuda_device
    p = CASES[name]
    case = ru.build_case(**p)
    fa, ours, grads, ours_b = run_ours(case, dev)
    so = ru.our_state(ours, case["P"], p["W"], p["H"])
    o = ru.oracle_for_case(case)
    oo = o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(), grads["invdepth"].numpy())
    assert ours[0] == oo["num_rendered"]
    assert np.array_equal(so["keys"].cpu().numpy().view(np.uint64), oo["keys"])
    assert np.array_equal(so["point_list"].cpu().numpy().view(np.uint32), oo["point_list"])
    assert np.array_equal(so["ranges"].cpu().numpy().view(np.uint32), oo["ranges"])
    assert np.array_equal(ours[2].cpu().numpy(), oo["radii"])
    # With ts/kids the reference evaluates pow with the GPU's approximate lg2/ex2 (forward.cu:550),
    # which libm cannot reproduce bit for bit: a handful of alpha ~ 1/255 decisions may flip.
    hier = p.get("with_hier", False)
    out = 16 if hier else 0
    assert int((so["n_contrib"].cpu().numpy().view(np.uint32) != oo["n_contrib"]).sum()) <= out
    assert int((ours[3].cpu().numpy() != oo["out_observe"]).sum()) <= out
    assert img_close(ours[1], oo["color"], max_outliers=out) and img_close(ours[4], oo["all_map"], atol=2e-4 if hier else IMG_ATOL, max_outliers=3 * out)
    assert img_close(ours[5], oo["plane_depth"], rtol=1e-4, max_outliers=out) and img_close(ours[9], oo["invdepth"], max_outliers=out)
    theirs = [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES]
    if hier:
        for a, b in zip(ours_b, theirs):
            assert ru.rel_report(a.cpu(), b)[2] < 2e-3
    else:
        ru.assert_grads_close([g.cpu() for g in ours_b], theirs, what=name)


# ------------------------------------------------------------------ variants
@pytest.mark.parametrize("render_geo,do_depth", [(False, False), (True, False), (False, True)])
def test_output_switches(cuda_device, render_geo, do_depth):
    dev = cuda_device
    case = ru.build_case(3000, 160, 96, seed=31)
    fa, ours, grads, ours_b = run_ours(case, dev, render_geo=render_geo, do_depth=do_depth)
    o = ru.oracle_for_case(case, render_geo=render_geo, do_depth=do_depth)
    oo = o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(),
                    grads["invdepth"].numpy() if do_depth else None)
    assert ours[9].shape == ((1 if do_depth else 0), 96, 160)
    assert img_close(ours[1], oo["color"]) and img_close(ours[4], oo["all_map"]) and img_close(ours[5], oo["plane_depth"], rtol=1e-4)
    if not render_geo:
        assert float(ours[4].abs().max()) == 0.0 and float(ours[5].abs().max()) == 0.0
    ru.assert_grads_close([g.cpu() for g in ours_b], [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES])


@pytest.mark.parametrize("degree", [0, 1, 2, 3])
def test_sh_degrees(cuda_device, degree):
    dev = cuda_device
    case = ru.build_case(2500, 128, 80, seed=40 + degree, sh_degree=degree)
    fa, ours, grads, ours_b = run_ours(case, dev)
    o = ru.oracle_for_case(case)
    oo = o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(), grads["invdepth"].numpy())
    assert img_close(ours[1], oo["color"])
    ru.assert_grads_close([g.cpu() for g in ours_b], [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES])
    k = (degree + 1) ** 2
    assert float(ours_b[5][:, k:, :].abs().max() if k < 16 else 0.0) == 0.0  # inactive bands get zero gradient


def test_precomputed_colors(cuda_device):
    dev = cuda_device
    case = ru.build_case(2500, 128, 80, seed=50)
    cols = torch.rand(case["P"], 3, generator=torch.Generator().manual_seed(5))
    fa, ours, grads, ours_b = run_ours(case, dev, colors_precomp=cols)
    o = ru.oracle_for_case(case, colors_precomp=cols)
    oo = o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(), grads["invdepth"].numpy())
    assert img_close(ours[1], oo["color"])
    assert ours_b[5].numel() == 0  # dL_dsh has shape (N, 0, 3)
    names = [n for n in ru.GRAD_NAMES if n != "dL_dsh"]
    ru.assert_grads_close([g.cpu() for n, g in zip(ru.GRAD_NAMES, ours_b) if n != "dL_dsh"],
                          [torch.from_numpy(og[n]) for n in names], names=names)


# ------------------------------------------------------------------ edge cases
def test_empty_inputs(cuda_device):
    dev = cuda_device
    case = ru.build_case(8, 64, 48, seed=60)
    for k in ("means3D", "scales", "rotations", "opacity", "shs", "all_map"):
        case[k] = case[k][:0].contiguous()
    case["P"] = 0
    fa, ours, grads, ours_b = run_ours(case, dev)
    assert ours[0] == 0 and ours[2].numel() == 0
    assert float(ours[1].abs().max()) == 0.0  # rasterize_points.cu:100: nothing rendered, zeros (not background)
    assert all(g.shape[0] == 0 for g in ours_b)


def test_everything_culled(cuda_device):
    dev = cuda_device
    case = ru.build_case(500, 64, 48, seed=61, eye=(0.0, 0.0, 50.0))  # scene is behind the camera
    fa, ours, grads, ours_b = run_ours(case, dev)
    assert ours[0] == 0 and int((ours[2] > 0).sum()) == 0
    assert float(ours[1].abs().max()) == 0.0  # rasterizer_impl.cu:332-333 returns before blending
    assert all(float(g.abs().max()) == 0.0 for g in ours_b if g.numel())


def test_single_instance_quirk(cuda_device):
    """R == 1: identifyTileRanges never closes the range (rasterizer_impl.cu:129-141) -> background only."""
    dev = cuda_device
    case = ru.build_case(1, 64, 48, seed=62)
    case["means3D"][:] = torch.tensor([[0.02, 0.02, 0.0]])
    case["scales"][:] = 1e-4
    case["all_map"] = syn.geometry_all_map(case["means3D"], case["scales"], case["rotations"], case["cam"])
    fa, ours, grads, ours_b = run_ours(case, dev)
    oo = ru.oracle_for_case(case).forward()
    assert ours[0] == oo["num_rendered"]
    assert img_close(ours[1], oo["color"])
    if ours[0] == 1:
        bg = torch.tensor([0.1, 0.2, 0.3], device=dev).view(3, 1, 1)
        assert torch.allclose(ours[1], bg.expand_as(ours[1]))


def test_debug_mode_and_repeatability(cuda_device):
    dev = cuda_device
    case = ru.build_case(3000, 160, 96, seed=63)
    fa = list(ru.op_args(case, dev))
    a = ru.OUR_C.rasterize_gaussians(*fa)
    fa[24] = True  # debug: synchronise + check after every launch
    b = ru.OUR_C.rasterize_gaussians(*fa)
    for i in (1, 2, 3, 4, 5, 9):
        assert torch.equal(a[i], b[i])  # the forward is deterministic, bit for bit


def test_mark_visible(cuda_device):
    dev = cuda_device
    case = ru.build_case(4000, 64, 48, seed=64, eye=(0.0, 0.0, -1.0))
    cam = case["cam"]
    from hidegs_b200.diff_gaussian_rasterization import GaussianRasterizer
    r = GaussianRasterizer(syn.raster_settings(cam, dev))
    vis = r.markVisible(case["means3D"].to(dev))
    W = cam.world_view_transform
    z = (case["means3D"] @ W[:3, 2] + W[3, 2])
    assert vis.dtype == torch.bool and int((vis.cpu() != (z > 0.2)).sum()) <= 2  # <=2: fp contraction at the threshold


# ------------------------------------------------------------------ public autograd API
def test_autograd_module_matches_operator(cuda_device):
    dev = cuda_device
    from hidegs_b200.diff_gaussian_rasterization import GaussianRasterizer
    case = ru.build_case(3000, 160, 96, seed=70)
    cam = case["cam"]
    rs = syn.raster_settings(cam, dev, bg=(0.1, 0.2, 0.3))
    t = {k: case[k].to(dev).requires_grad_(True) for k in ("means3D", "shs", "opacity", "scales", "rotations", "all_map")}
    means2D = torch.zeros_like(t["means3D"], requires_grad=True)
    color, radii, observe, all_map, plane_depth, invdepth = GaussianRasterizer(rs)(
        means3D=t["means3D"], means2D=means2D, opacities=t["opacity"], shs=t["shs"], scales=t["scales"],
        rotations=t["rotations"], all_map=t["all_map"])
    g = {k: v.to(dev) for k, v in syn.upstream_grads(160, 96).items()}
    loss = (color * g["color"]).sum() + (all_map * g["all_map"]).sum() + (plane_depth * g["plane_depth"]).sum() + (invdepth * g["invdepth"]).sum()
    loss.backward()
    fa, fwd, grads, bwd = run_ours(case, dev)
    named = dict(zip(ru.GRAD_NAMES, bwd))
    ru.assert_grads_close([means2D.grad, t["opacity"].grad, t["means3D"].grad, t["shs"].grad, t["scales"].grad, t["rotations"].grad, t["all_map"].grad],
                          [named[n] for n in ("dL_dmeans2D", "dL_dopacity", "dL_dmeans3D", "dL_dsh", "dL_dscales", "dL_drotations", "dL_dall_map")],
                          names=("means2D", "opacity", "means3D", "sh", "scales", "rotations", "all_map"))
    assert not radii.requires_grad and not observe.requires_grad


# ------------------------------------------------------------------ full size (BASELINE config 2)
def test_full_size_properties(cuda_device):
    """1M Gaussians, 1920x1080, SH degree 3: size-independent properties of the binning and the blend."""
    dev = cuda_device
    W, H, n = 1920, 1080, 1_000_000
    case = ru.build_case(n, W, H, seed=0)
    fa, ours, grads, bwd = run_ours(case, dev)
    so = ru.our_state(ours, n, W, H)
    R = ours[0]
    assert R == int(so["tiles_touched"].long().sum()) and R > n
    keys = so["keys"]
    assert bool((keys[1:] >= keys[:-1]).all())  # sortedness
    assert torch.equal(keys.sort()[0], so["keys_unsorted"].sort()[0])  # the sort is a permutation
    # values follow their keys: recompute each key from its value
    pl = so["point_list"].long()
    depth_bits = so["depths"].view(torch.int32)[pl].long() & 0xFFFFFFFF
    assert torch.equal(keys & 0xFFFFFFFF, depth_bits)
    # tile ranges partition [0, R)
    rg = so["ranges"].long()
    nz = rg[rg[:, 1] > rg[:, 0]]
    assert int((nz[:, 1] - nz[:, 0]).sum()) == R and int(nz[0, 0]) == 0 and int(nz[-1, 1]) == R
    assert torch.equal(nz[1:, 0], nz[:-1, 1])
    tiles = (keys >> 32)
    assert torch.equal(tiles[nz[:, 0]], torch.arange(rg.shape[0], device=dev)[rg[:, 1] > rg[:, 0]])
    # blend: transmittance in (0,1], n_contrib inside its range, colour = C + T*bg bounded
    assert float(so["final_T"].min()) > 0.0 and float(so["final_T"].max()) <= 1.0
    assert all(bool(torch.isfinite(ours[i]).all()) for i in (1, 4, 9))
    # stable tie order: equal keys keep ascending slot order
    same = keys[1:] == keys[:-1]
    assert bool((pl[1:][same] > pl[:-1][same]).all())
    # backward is linear in the upstream gradient
    g2 = {k: 2.0 * v for k, v in grads.items()}
    bwd2 = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, ours, g2, dev))
    ru.assert_grads_close(bwd2, [2.0 * g for g in bwd], what="linearity")
    # culled Gaussians receive exactly zero gradient
    dead = ours[2] <= 0
    assert all(float(g[dead].abs().max()) == 0.0 for g in bwd if g.numel())
    if ru.ref_available():
        REF = ru.ref_module()
        ref = REF.rasterize_gaussians(*fa)
        sr = ru.ref_state(ref, n, W, H)
        assert ref[0] == R
        for k in ("keys", "point_list", "ranges", "n_contrib"):
            assert torch.equal(so[k], sr[k]), k
        assert img_close(ours[1], ref[1]) and img_close(ours[9], ref[9])
        ref_b = REF.rasterize_gaussians_backward(*ru.bwd_args(fa, ref, grads, dev))
        ru.assert_grads_close(bwd, ref_b, what="config2 vs reference")


# ------------------------------------------------------------------ full size (BASELINE config 3)
def test_config3_uav_4k_lod_cut(cuda_device):
    """configs[2]: 6M Gaussians on the UAV slab, 3840x2160 nadir view, synthetic hierarchy cut (60 % of the nodes,
    random parents, half of the interpolation weights exactly 1, 2..8 kids), rendered the way render_post does it
    (Python interpolation with the parent, then the rasterizer with weights / kid counts, no geometry, no depth) and,
    additionally, through the raw indices / parent_indices API — ours vs the UNMODIFIED reference on the same inputs."""
    import math
    dev = cuda_device
    W, H, n = 3840, 2160, 6_000_000
    sc = syn.make_uav_scene(n, seed=0)
    cam = syn.look_at_camera((0.0, 0.0, 120.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), math.radians(70.0), W, H)
    g = torch.Generator().manual_seed(5)
    keep = (torch.rand(n, generator=g) < 0.6).nonzero().flatten()
    P = keep.numel()
    rest = torch.ones(n, dtype=torch.bool)
    rest[keep] = False
    rest = rest.nonzero().flatten()
    parents = rest[torch.randint(0, rest.numel(), (P,), generator=g)]
    ts = torch.rand(P, generator=g)
    ts[torch.rand(P, generator=g) < 0.5] = 1.0
    kids = torch.randint(2, 9, (P,), generator=g, dtype=torch.int32)
    d = {k: v.to(dev) for k, v in sc.items()}
    keep_d, par_d, ts_d, kids_d = keep.to(dev), parents.to(dev), ts.to(dev), kids.to(dev)
    e_i = torch.empty(0, dtype=torch.int32, device=dev)
    e_f = torch.empty(0, dtype=torch.float32, device=dev)
    bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    camd = cam.to(dev)

    # ---- path A: render_post semantics (gaussian_renderer/__init__.py:278-324)
    t1, t0 = ts_d[:, None], (1 - ts_d)[:, None]
    m3 = (t1 * d["means3D"][keep_d] + t0 * d["means3D"][par_d]).contiguous()
    scl = (t1 * d["scales"][keep_d] + t0 * d["scales"][par_d]).contiguous()
    shs = (t1[:, :, None] * d["shs"][keep_d] + t0[:, :, None] * d["shs"][par_d]).contiguous()
    rp, rc = d["rotations"][par_d].clone(), d["rotations"][keep_d]
    rp[(rc * rp).sum(1) < 0] *= -1
    rot = (t1 * rc + t0 * rp).contiguous()
    op = (t1 * d["opacity"][keep_d] + t0 * d["opacity"][par_d]).contiguous()
    fa = (bg, e_i, e_i, ts_d, kids_d, m3, e_f, e_f, op, scl, rot, 1.0, e_f, camd.world_view_transform,
          camd.full_proj_transform, cam.tanfovx, cam.tanfovy, H, W, shs, 3, camd.camera_center, False, False, False, False)
    ours = ru.OUR_C.rasterize_gaussians(*fa)
    R = ours[0]
    assert R > 0 and int((ours[2] > 0).sum()) > 100_000
    gr = dict(color=torch.randn(3, H, W, generator=g).to(dev), all_map=torch.zeros(5, H, W, device=dev),
              plane_depth=torch.zeros(1, H, W, device=dev), invdepth=torch.zeros(0, H, W, device=dev))
    ours_b = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, ours, gr, dev))
    so = ru.our_state(ours, P, W, H)
    keys = so["keys"]
    assert bool((keys[1:] >= keys[:-1]).all()) and int(so["tiles_touched"].long().sum()) == R
    assert int((keys >> 32).max()) < 240 * 135
    if ru.ref_available():
        REF = ru.ref_module()
        ref = REF.rasterize_gaussians(*fa)
        sr = ru.ref_state(ref, P, W, H)
        assert ref[0] == R
        for k in ("keys", "point_list", "ranges", "n_contrib"):
            assert torch.equal(so[k], sr[k]), k
        assert torch.equal(ours[2], ref[2]) and torch.equal(ours[3], ref[3])
        assert img_close(ours[1], ref[1])
        ref_b = REF.rasterize_gaussians_backward(*ru.bwd_args(fa, ref, gr, dev))
        ru.assert_grads_close(ours_b, ref_b, what="config3 render_post path", max_bad_frac=1e-6)
        del ref, ref_b, sr
    del ours, ours_b, so, keys

    # ---- path B: the raw API (indices / parent_indices inside the rasterizer), smaller image to bound the run time
    W2, H2 = 1920, 1080
    cam2 = syn.look_at_camera((0.0, 0.0, 120.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), math.radians(70.0), W2, H2).to(dev)
    fb = (bg, keep_d.int(), par_d.int(), ts_d, kids_d, d["means3D"], e_f, e_f, d["opacity"], d["scales"], d["rotations"], 1.0,
          e_f, cam2.world_view_transform, cam2.full_proj_transform, cam2.tanfovx, cam2.tanfovy, H2, W2, d["shs"], 0,
          cam2.camera_center, False, False, False, False)
    ours = ru.OUR_C.rasterize_gaussians(*fb)
    gr2 = dict(color=torch.randn(3, H2, W2, generator=g).to(dev), all_map=torch.zeros(5, H2, W2, device=dev),
               plane_depth=torch.zeros(1, H2, W2, device=dev), invdepth=torch.zeros(0, H2, W2, device=dev))
    ours_b = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fb, ours, gr2, dev))
    if ru.ref_available():
        ref = REF.rasterize_gaussians(*fb)
        assert ref[0] == ours[0]
        so, sr = ru.our_state(ours, P, W2, H2), ru.ref_state(ref, P, W2, H2)
        for k in ("keys", "point_list", "ranges", "n_contrib"):
            assert torch.equal(so[k], sr[k]), k
        assert img_close(ours[1], ref[1])
        ref_b = REF.rasterize_gaussians_backward(*ru.bwd_args(fb, ref, gr2, dev))
        # SH degree 0: the parent rows are fully defined (see mask_undefined_parent_rows)
        ru.assert_grads_close(ours_b, ref_b, what="config3 raw indices path", max_bad_frac=1e-6)

    # ---- scale regularisation on the visible set (frequency_regularization.py:1403-1444) vs the oracle
    from hidegs_b200.frequency_regularization import _ScaleReg
    import oracle.loss_oracle as lo
    vis = (ours[2] > 0).nonzero().flatten()
    s_gpu = d["scales"].clone().requires_grad_(True)
    v_gpu = _ScaleReg.apply(s_gpu, keep_d[vis])
    v_gpu.backward()
    s_cpu = sc["scales"].clone().requires_grad_(True)
    v_cpu = lo.scale_regularization(s_cpu, keep[vis.cpu()])
    v_cpu.backward()
    assert abs(v_gpu.item() - v_cpu.item()) <= 1e-5 * abs(v_cpu.item()) + 1e-12
    ru.assert_grads_close([s_gpu.grad], [s_cpu.grad], names=("scaling",), what="scale regularisation")


def test_sh_gradient_sink_and_chunked_backward(cuda_device):
    """Extensions of the backward: the SH gradient accumulated into a caller-owned sink (beta 0 / 1, culled rows left
    alone) and the per-Gaussian part issued in slot ranges with a hook per range — same gradients as the plain call."""
    from hidegs_b200 import synthetic as syn
    dev = cuda_device
    case = ru.build_case(9000, 176, 112, seed=21)
    fa = ru.op_args(case, dev)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    grads = syn.upstream_grads(176, 112)
    ba = ru.bwd_args(fa, fwd, grads, dev)
    plain = [g.clone() for g in ru.OUR_C.rasterize_gaussians_backward(*ba)]
    dead = fwd[2] == 0
    assert 0 < int(dead.sum()) < dead.numel()
    # beta = 0: the sink is overwritten (culled rows zero-filled), dL_dsh comes back as None
    sink = torch.full_like(plain[5], 7.0)
    out = ru.OUR_C.rasterize_gaussians_backward(*ba, sh_sink=(sink, 0.0))
    assert out[5] is None
    ru.assert_grads_close([sink], [plain[5]], names=("dL_dsh",), what="sink beta=0")
    assert float(sink[dead].abs().max()) == 0.0
    for i in (0, 1, 2, 3, 4, 6, 7, 8):
        ru.assert_grads_close([out[i]], [plain[i]], names=(ru.GRAD_NAMES[i],), what="sink other grads")
    # beta = 1: accumulated on top; rows of culled Gaussians are not touched (bit for bit)
    base = torch.randn_like(plain[5])
    sink = base.clone()
    ru.OUR_C.rasterize_gaussians_backward(*ba, sh_sink=(sink, 1.0))
    assert torch.equal(sink[dead], base[dead])
    ru.assert_grads_close([sink - base], [plain[5]], names=("dL_dsh",), what="sink beta=1", l2_tol=1e-3, rtol=5e-3)
    # chunked: ranges are multiples of 128 slots, cover every slot once, and the gradients are the same
    seen = []
    chunked = ru.OUR_C.rasterize_gaussians_backward(*ba, chunk_hook=(4, lambda c, p0, p1: seen.append((c, p0, p1))))
    with pytest.raises(ZeroDivisionError):  # an exception raised inside the hook surfaces after the C frame returns
        ru.OUR_C.rasterize_gaussians_backward(*ba, chunk_hook=(2, lambda c, p0, p1: 1 // 0))
    assert [c for c, _, _ in seen] == list(range(len(seen))) and 2 <= len(seen) <= 4
    assert seen[0][1] == 0 and seen[-1][2] == 9000 and all(a[2] == b[1] for a, b in zip(seen, seen[1:]))
    assert all(p0 % 128 == 0 for _, p0, _ in seen)
    ru.assert_grads_close(chunked, plain, what="chunked backward")
    # an index remap cannot feed a sink
    with pytest.raises(RuntimeError, match="sink"):
        hier = ru.build_case(3000, 96, 64, seed=3, with_indices=True, with_hier=True)
        fh = ru.op_args(hier, dev)
        fw = ru.OUR_C.rasterize_gaussians(*fh)
        gh = syn.upstream_grads(96, 64)
        bh = ru.bwd_args(fh, fw, gh, dev)
        ru.OUR_C.rasterize_gaussians_backward(*bh, sh_sink=(torch.zeros(hier["means3D"].shape[0], 16, 3, device=dev), 0.0))


# (degree, SH coefficients M): rows of 3 M floats that are not a multiple of 4 take the per-thread paths of both kernels
@pytest.mark.parametrize("degree,M", [pytest.param(3, 16, id="3"), pytest.param(1, 16, id="1"),
                                      pytest.param(0, 1, id="0-M1"), pytest.param(1, 9, id="1-M9"),
                                      pytest.param(2, 15, id="2-M15")])
def test_sh_gradient_factors_rebuild_the_summed_rows(cuda_device, degree, M):
    """Factored exchange (include/hidegs_exchange.h): with `sh_factor` the backward writes three colour-gradient factors
    per Gaussian + the camera centre instead of the SH rows; hg_sh_gradient_from_factors over the blocks of several
    views rebuilds exactly the sum of the rows the plain backward writes for those views; every other gradient is
    untouched."""
    from hidegs_b200 import parallel, synthetic as syn
    dev = cuda_device
    N, W, H = 9000, 176, 112
    eyes = [(0.0, 0.0, -5.0), (1.5, 0.4, -4.5), (-2.0, -0.6, -4.0)]
    block = 3 * N + 4
    factors = torch.full((len(eyes) * block,), 3.0, device=dev)
    want = None
    some_dead = False
    for v, eye in enumerate(eyes):
        case = ru.build_case(N, W, H, seed=21, sh_degree=degree, eye=eye, sh_coeffs=M)
        fa = ru.op_args(case, dev)
        fwd = ru.OUR_C.rasterize_gaussians(*fa)
        ba = ru.bwd_args(fa, fwd, syn.upstream_grads(W, H, seed=v), dev)
        plain = [g.clone() for g in ru.OUR_C.rasterize_gaussians_backward(*ba)]
        mine = factors[v * block:(v + 1) * block]
        out = ru.OUR_C.rasterize_gaussians_backward(*ba, sh_factor=mine)
        assert out[5] is None
        for i in (0, 1, 2, 3, 4, 6, 7, 8):
            ru.assert_grads_close([out[i]], [plain[i]], names=(ru.GRAD_NAMES[i],), what="factor mode, other grads")
        dead = fwd[2] == 0
        some_dead |= bool(dead.any())
        assert float(mine[:3 * N].view(N, 3)[dead].abs().max()) == 0.0          # culled slots: zero factors
        assert torch.equal(mine[3 * N:3 * N + 3], fa[21])                       # the view's camera centre rides along
        # one view alone: the rebuilt rows are the plain rows (up to the FMA contraction of the basis polynomials)
        single = torch.full_like(plain[5], 9.0)
        parallel.sh_gradient_from_factors(fa[5], mine, 1, block, degree, single, beta=0.0)
        ru.assert_grads_close([single], [plain[5]], names=("dL_dsh",), what="rebuilt rows, one view", l2_tol=1e-6, rtol=1e-5)
        assert float(single[dead].abs().max()) == 0.0
        want = plain[5].double() if want is None else want + plain[5].double()
        means3D = fa[5]
    assert some_dead
    got = torch.full_like(plain[5], -1.0)
    parallel.sh_gradient_from_factors(means3D, factors, len(eyes), block, degree, got, beta=0.0)
    ru.assert_grads_close([got], [want.float()], names=("dL_dsh",), what="rebuilt sum", l2_tol=1e-6, rtol=1e-5)
    acc = got.clone()
    parallel.sh_gradient_from_factors(means3D, factors, len(eyes), block, degree, acc, beta=1.0)
    ru.assert_grads_close([acc], [(2 * want).float()], names=("dL_dsh",), what="rebuilt sum, beta=1", l2_tol=1e-6, rtol=1e-5)
    with pytest.raises(RuntimeError, match="factors"):  # an index remap cannot be factored
        hier = ru.build_case(3000, 96, 64, seed=3, with_indices=True, with_hier=True)
        fh = ru.op_args(hier, dev)
        fw = ru.OUR_C.rasterize_gaussians(*fh)
        bh = ru.bwd_args(fh, fw, syn.upstream_grads(96, 64), dev)
        ru.OUR_C.rasterize_gaussians_backward(*bh, sh_factor=torch.zeros(3 * hier["means3D"].shape[0] + 4, device=dev))


@pytest.mark.parametrize("degree", [3, 2])
def test_sparse_view_zero_rows(cuda_device, degree):
    """A view that culls most Gaussians (R < 2 P): the zero rows of culled slots come from memsets, live rows from the
    kernel — every gradient row must be defined even when the arena starts as NaN (degree 2: per-thread SH path)."""
    from hidegs_b200 import synthetic as syn
    dev = cuda_device
    case = ru.build_case(8000, 96, 64, seed=9 + degree, sh_degree=degree, eye=(4.5, 0.0, -5.0))
    fa = ru.op_args(case, dev)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    assert 0 < fwd[0] < 2 * 8000 and int((fwd[2] > 0).sum()) < 4000
    grads = syn.upstream_grads(96, 64)
    poisoned = torch.full((8000 * 84,), float("nan"), device=dev)  # caller-owned arena (>= 80 floats per Gaussian)
    ours_b = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, fwd, grads, dev), grad_arena=poisoned)
    assert ours_b[3].data_ptr() == poisoned.data_ptr()  # the gradients are views of the arena
    assert all(bool(torch.isfinite(g).all()) for g in ours_b)
    o = ru.oracle_for_case(case)
    o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(), grads["invdepth"].numpy())
    ru.assert_grads_close([g.cpu() for g in ours_b], [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES], what="sparse view")
    dead = (fwd[2] == 0).cpu()
    assert all(float(g.cpu()[dead].abs().max()) == 0.0 for g in ours_b)
