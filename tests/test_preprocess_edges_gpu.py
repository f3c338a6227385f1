"""Edge cases of the rasterizer's per-Gaussian passes, preprocess_fwd (csrc/preprocess.cu) and preprocess_bwd
(csrc/preprocess_bwd.cu), on the B200: every SH width the API accepts, misaligned contiguous views, the covariance
source and scale modifier, and the projection edges.

Every case is held to two references:
  * the CPU oracle (oracle/raster_oracle.c) with the criteria of test_raster_gpu.test_parity_vs_cpu_oracle: tile keys,
    sorted list, tile ranges and radii exact, images within 1e-4, gradients within ru.assert_grads_close;
  * a float64 restatement of the per-Gaussian colour and its SH backward (below): the colour of every visible slot from
    its SH row and view direction, and dL/dSH = basis x clamp-masked dL/dRGB from the same run's dL_dcolors.  This
    part of the backward involves no atomics, so it is exact up to float32 rounding.

The scenes put culled slots between live ones inside every warp (every third mean behind the camera, a random tenth
off screen), and have N = 3001 slots, which is not a multiple of 32 or of the 128-slot CTA.
"""
import math

import numpy as np
import pytest
import torch

import raster_utils as ru
from hidegs_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

N = 3001
IMG_ATOL = 1e-4
# Colour (record rgb) vs float64, absolute; dL/dSH vs float64, relative to its largest entry.  Largest errors measured
# over every case of this file on an NVIDIA B200 (power limit 1000 W): rgb 1.8e-7, 1/depth 8.9e-8 relative, dL/dSH
# 2.4e-7 of the maximum (the flat-Gaussian case).
RGB_ATOL = 2e-6
INVDEPTH_RTOL = 1e-6
DSH_RTOL_OF_MAX = 1e-6
PRE_CLAMP_EXCLUDE = 1e-6  # entries whose pre-clamp colour lies this close to 0 may take either side of the clamp

SH_C0 = 0.28209479177387814
SH_C1 = 0.4886025119029199
SH_C2 = (1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792, 0.5462742152960396)
SH_C3 = (-0.5900435899266435, 2.890611442640554, -0.4570457994644658, 0.3731763325901154, -0.4570457994644658,
         1.445305721320277, -0.5900435899266435)


# ------------------------------------------------------------------ scenes
def edge_scene(M, D, seed, W=160, H=96, n=N):
    """ru.build_case with M SH coefficients, where culled slots sit between live ones inside every warp."""
    case = ru.build_case(n, W, H, seed=seed, sh_degree=D, sh_coeffs=M)
    g = torch.Generator().manual_seed(seed + 7)
    m = case["means3D"]
    m[::3, 2] = -6.0  # behind the camera (eye at z = -5 looking down +z)
    off = torch.rand(n, generator=g) < 0.1
    m[off, 0] = torch.where(m[off, 0] >= 0, 40.0, -40.0)  # in front of the camera, far outside the image
    refresh_all_map(case)
    return case


def refresh_all_map(case):
    case["all_map"] = syn.geometry_all_map(case["means3D"], case["scales"], case["rotations"], case["cam"])


def view_to_world(xv, yv, zv):
    """The default camera has no rotation: world = view - (0, 0, 5)."""
    return torch.stack([xv, yv, zv - 5.0], 1)


def run(case, dev, scale_modifier=1.0, cov3D=None, shs=None, rotations=None):
    """Forward + backward through the torch extension; `shs` / `rotations` replace the case's tensors (e.g. views)."""
    e_f = torch.empty(0, dtype=torch.float32, device=dev)
    fa = list(ru.op_args(case, dev))
    fa[11] = scale_modifier
    if cov3D is not None:
        fa[9], fa[10], fa[12] = e_f, e_f, cov3D.to(dev)
    if shs is not None:
        fa[19] = shs
    if rotations is not None:
        fa[10] = rotations
    fa = tuple(fa)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    grads = syn.upstream_grads(case["W"], case["H"])
    bwd = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, fwd, grads, dev))
    torch.cuda.synchronize()
    return fa, fwd, grads, bwd


def max_abs_diff(a, b):
    return float((torch.as_tensor(a).double().cpu() - torch.as_tensor(b).double().cpu()).abs().max())


def check_vs_oracle(case, fwd, grads, bwd, what, **oracle_kw):
    """The criteria of test_parity_vs_cpu_oracle (no hierarchy inputs: no outliers allowed)."""
    so = ru.our_state(fwd, case["P"], case["W"], case["H"])
    o = ru.oracle_for_case(case, nthreads=8, **oracle_kw)
    oo = o.forward()
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(),
                    grads["invdepth"].numpy())
    assert fwd[0] == oo["num_rendered"] and fwd[0] > 0, (what, fwd[0], oo["num_rendered"])
    assert np.array_equal(so["keys"].cpu().numpy().view(np.uint64), oo["keys"]), what
    assert np.array_equal(so["point_list"].cpu().numpy().view(np.uint32), oo["point_list"]), what
    assert np.array_equal(so["ranges"].cpu().numpy().view(np.uint32), oo["ranges"]), what
    assert np.array_equal(fwd[2].cpu().numpy(), oo["radii"]), what
    for i, name in ((1, "color"), (4, "all_map"), (9, "invdepth")):
        err = max_abs_diff(fwd[i], oo[name])
        assert err <= IMG_ATOL, "%s: %s differs from the oracle by %.3g" % (what, name, err)
    pd_ours, pd_oracle = fwd[5].double().cpu(), torch.from_numpy(oo["plane_depth"]).double()
    assert bool(((pd_ours - pd_oracle).abs() <= IMG_ATOL + 1e-4 * pd_oracle.abs()).all()), what
    ru.assert_grads_close([g.cpu() for g in bwd], [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES], what=what)
    return so


# ------------------------------------------------------------------ float64 restatement
def sh_basis64(dirs, D):
    """[n, (D+1)^2] SH basis of computeColorFromSH (forward.cu:25-76) at the normalised directions, float64."""
    d = dirs / dirs.norm(dim=1, keepdim=True)
    x, y, z = d.unbind(1)
    b = [torch.full_like(x, SH_C0)]
    if D > 0:
        b += [-SH_C1 * y, SH_C1 * z, -SH_C1 * x]
    if D > 1:
        xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
        b += [SH_C2[0] * xy, SH_C2[1] * yz, SH_C2[2] * (2 * zz - xx - yy), SH_C2[3] * xz, SH_C2[4] * (xx - yy)]
    if D > 2:
        b += [SH_C3[0] * y * (3 * xx - yy), SH_C3[1] * xy * z, SH_C3[2] * y * (4 * zz - xx - yy),
              SH_C3[3] * z * (2 * zz - 3 * xx - 3 * yy), SH_C3[4] * x * (4 * zz - xx - yy), SH_C3[5] * z * (xx - yy),
              SH_C3[6] * x * (xx - 3 * yy)]
    return torch.stack(b, 1)


class ColourChain:
    """Per-slot colour, inverse depth and SH-gradient factors of one forward, restated in float64."""

    def __init__(self, case, fwd):
        self.D = case["sh_degree"]
        self.nb = (self.D + 1) ** 2
        self.live = (fwd[2] > 0).cpu()
        assert int(self.live.sum()) > 0
        cam = case["cam"]
        m = case["means3D"].double()[self.live]
        sh = case["shs"].double()[self.live][:, :self.nb, :]
        self.basis = sh_basis64(m - cam.camera_center.double(), self.D)              # [L, nb]
        self.pre = torch.einsum("lk,lkc->lc", self.basis, sh) + 0.5                   # colour before the clamp
        V = cam.world_view_transform.double()                                        # transposed view matrix
        self.depth = m @ V[:3, 2] + V[3, 2]
        self.so = ru.our_state(fwd, case["P"], case["W"], case["H"])

    def check_forward(self, what):
        rec = self.so["records"].cpu().double()[self.live]
        err_rgb = float((rec[:, 6:9] - self.pre.clamp_min(0.0)).abs().max())
        err_invd = float(((rec[:, 9] - 1.0 / self.depth) * self.depth).abs().max())
        print("%s: rgb max err %.3g, 1/depth max rel err %.3g" % (what, err_rgb, err_invd))
        assert err_rgb <= RGB_ATOL, "%s: record rgb differs from float64 by %.3g" % (what, err_rgb)
        assert err_invd <= INVDEPTH_RTOL, "%s: record 1/depth differs from float64 by %.3g (relative)" % (what, err_invd)

    def want_dsh(self, dL_dcolors):
        """dL/dSH[g, k, c] = basis_k * dL_dcolors[g, c] * [pre-clamp colour >= 0], and the mask of decidable entries."""
        dcol = dL_dcolors.detach().cpu().double()[self.live]
        want = self.basis[:, :, None] * (dcol * (self.pre >= 0))[:, None, :]
        ok = (self.pre.abs() > PRE_CLAMP_EXCLUDE)[:, None, :].expand_as(want)
        return want, ok

    def check_dsh(self, dL_dsh, dL_dcolors, what, base=None):
        """dL_dsh [N, M, 3] (minus `base` where it was accumulated onto it) against the float64 chain; bands above
        the degree and the rows of culled slots exactly zero."""
        want, ok = self.want_dsh(dL_dcolors)
        got = dL_dsh.detach().cpu().double()
        if base is not None:
            got = got - base.detach().cpu().double()
        scale = float(want.abs().max())
        assert scale > 0.0
        err = float(((got[self.live][:, :self.nb, :] - want).abs() * ok).max())
        print("%s: dL/dSH max err %.3g of max %.3g (%.3g)" % (what, err, scale, err / scale))
        assert err <= DSH_RTOL_OF_MAX * scale, "%s: dL/dSH differs from float64 by %.3g of its max" % (what, err / scale)
        assert float(got[:, self.nb:, :].abs().max() if got.shape[1] > self.nb else 0.0) == 0.0, what
        assert float(got[~self.live].abs().max()) == 0.0, what
        return scale


def interleaved_rows(fwd):
    """Live slots whose predecessor in the same warp is culled."""
    live = (fwd[2] > 0).cpu()
    idx = torch.arange(1, live.numel())
    return int((live[1:] & ~live[:-1] & (idx % 32 != 0)).sum())


# ------------------------------------------------------------------ SH width x degree
SH_WIDTHS = [(1, 0), (3, 0), (4, 1), (9, 1), (9, 2), (15, 2), (16, 0), (16, 3)]


@pytest.mark.parametrize("M,D", SH_WIDTHS, ids=["M%d-D%d" % md for md in SH_WIDTHS])
def test_sh_width_and_degree(cuda_device, M, D):
    """Any SH width M in 1..16 (3 M floats per row; only 4 | 3 M lets a row start on a float4) at degrees up to the
    widest that fits, forward and backward; with 4 | 3 M also the SH gradient sink at beta 0 and 1."""
    dev = cuda_device
    what = "M=%d D=%d" % (M, D)
    case = edge_scene(M, D, seed=100 + 4 * M + D)
    fa, fwd, grads, bwd = run(case, dev)
    assert interleaved_rows(fwd) > 300, what
    check_vs_oracle(case, fwd, grads, bwd, what)
    chain = ColourChain(case, fwd)
    chain.check_forward(what)
    scale = chain.check_dsh(bwd[5], bwd[1], what)

    sink_ok = (3 * M) % 4 == 0
    assert ru.OUR_C.sh_sink_supported(fa[19]) == sink_ok
    if not sink_ok:
        return
    ba = ru.bwd_args(fa, fwd, grads, dev)
    # beta = 0: the sink is overwritten, culled rows zero-filled
    sink = torch.full_like(bwd[5], 7.0)
    out = ru.OUR_C.rasterize_gaussians_backward(*ba, sh_sink=(sink, 0.0))
    assert out[5] is None
    chain.check_dsh(sink, out[1], what + " sink beta=0")
    # beta = 1: accumulated onto the sink (|base| <= max |dL/dSH| keeps the rounding of the sum below the bound);
    # rows of culled slots are not touched
    g = torch.Generator(device=dev).manual_seed(M)
    base = (torch.rand(bwd[5].shape, generator=g, device=dev) * 2 - 1) * scale
    sink = base.clone()
    out = ru.OUR_C.rasterize_gaussians_backward(*ba, sh_sink=(sink, 1.0))
    dead = fwd[2] <= 0
    assert torch.equal(sink[dead], base[dead])
    chain.check_dsh(sink, out[1], what + " sink beta=1", base=base)


def test_degree0_model_through_the_public_rasterizer(cuda_device):
    """A degree-0 model (features [N, 1, 3]) through GaussianRasterizer and autograd, against the oracle."""
    dev = cuda_device
    from hidegs_b200.diff_gaussian_rasterization import GaussianRasterizer
    case = edge_scene(1, 0, seed=150)
    cam = case["cam"]
    rs = syn.raster_settings(cam, dev, sh_degree=0, bg=(0.1, 0.2, 0.3))
    t = {k: case[k].to(dev).requires_grad_(True) for k in ("means3D", "shs", "opacity", "scales", "rotations", "all_map")}
    means2D = torch.zeros_like(t["means3D"], requires_grad=True)
    color, radii, observe, all_map, plane_depth, invdepth = GaussianRasterizer(rs)(
        means3D=t["means3D"], means2D=means2D, opacities=t["opacity"], shs=t["shs"], scales=t["scales"],
        rotations=t["rotations"], all_map=t["all_map"])
    g = syn.upstream_grads(case["W"], case["H"])
    gd = {k: v.to(dev) for k, v in g.items()}
    loss = ((color * gd["color"]).sum() + (all_map * gd["all_map"]).sum() + (plane_depth * gd["plane_depth"]).sum()
            + (invdepth * gd["invdepth"]).sum())
    loss.backward()
    o = ru.oracle_for_case(case, nthreads=8)
    oo = o.forward()
    og = o.backward(g["color"].numpy(), g["all_map"].numpy(), g["plane_depth"].numpy(), g["invdepth"].numpy())
    assert np.array_equal(radii.cpu().numpy(), oo["radii"])
    for name, ours in (("color", color), ("all_map", all_map), ("invdepth", invdepth)):
        err = max_abs_diff(ours.detach(), oo[name])
        assert err <= IMG_ATOL, "degree-0 model: %s differs from the oracle by %.3g" % (name, err)
    ru.assert_grads_close(
        [means2D.grad, t["opacity"].grad, t["means3D"].grad, t["shs"].grad, t["scales"].grad, t["rotations"].grad,
         t["all_map"].grad],
        [torch.from_numpy(og[n]) for n in ("dL_dmeans2D", "dL_dopacity", "dL_dmeans3D", "dL_dsh", "dL_dscales",
                                           "dL_drotations", "dL_dall_map")],
        names=("means2D", "opacity", "means3D", "sh", "scales", "rotations", "all_map"), what="degree-0 model")


# ------------------------------------------------------------------ misaligned views
def offset_view(t):
    """A contiguous copy of `t` that starts one float past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


def test_misaligned_sh_view(cuda_device):
    """SH rows in a contiguous view one float off a 16-byte boundary (M = 16): the forward stages them into shared memory
    float by float instead of by float4 and evaluates the same eval_sh on the same values, so every output is
    bit-identical to the aligned copy's.  The backward takes its per-thread SH path, which matches the float64 chain."""
    dev = cuda_device
    case = edge_scene(16, 3, seed=160)
    shs = offset_view(case["shs"].to(dev))
    assert not ru.OUR_C.sh_sink_supported(shs)
    _, fwd_a, _, _ = run(case, dev)
    fa, fwd, grads, bwd = run(case, dev, shs=shs)
    assert fwd[0] == fwd_a[0]
    for i in (1, 2, 3, 4, 5, 9):
        assert torch.equal(fwd[i], fwd_a[i]), i
    live = fwd[2] > 0
    rec = ru.our_state(fwd, case["P"], case["W"], case["H"])["records"][live]
    rec_a = ru.our_state(fwd_a, case["P"], case["W"], case["H"])["records"][live]
    assert torch.equal(rec.view(torch.int32), rec_a.view(torch.int32))
    check_vs_oracle(case, fwd, grads, bwd, "misaligned shs")
    chain = ColourChain(case, fwd)
    chain.check_forward("misaligned shs")
    chain.check_dsh(bwd[5], bwd[1], "misaligned shs")


def test_misaligned_rotations_view(cuda_device):
    """Rotations in a contiguous view one float off a 16-byte boundary: the library refuses such a pointer (its
    kernels read one float4 per row), the torch extension copies the view into aligned storage, and the results are
    those of the aligned tensor."""
    dev = cuda_device
    case = edge_scene(16, 3, seed=170)
    rot = offset_view(case["rotations"].to(dev))
    _, fwd_a, _, bwd_a = run(case, dev)
    fa, fwd, grads, bwd = run(case, dev, rotations=rot)
    assert fwd[0] == fwd_a[0]
    for i in (1, 2, 3, 4, 5, 9):
        assert torch.equal(fwd[i], fwd_a[i]), i
    ru.assert_grads_close([g.cpu() for g in bwd], [g.cpu() for g in bwd_a], what="misaligned rotations vs aligned")
    check_vs_oracle(case, fwd, grads, bwd, "misaligned rotations")


# ------------------------------------------------------------------ covariance source and scale modifier
def cov3d64(scales, rotations):
    """Upper triangle of R diag(s^2) R^T in float64 (build_covariance_from_scaling_rotation), rounded to fp32."""
    q = rotations.double()
    R = syn.quaternion_to_matrix(q / q.norm(dim=1, keepdim=True))
    L = R * scales.double()[:, None, :]
    S = L @ L.transpose(1, 2)
    return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1).float().contiguous()


@pytest.mark.parametrize("source", ["scale_modifier_0.5", "scale_modifier_1.7", "cov3D_precomp"])
def test_covariance_source_and_scale_modifier(cuda_device, source):
    """scale_modifier != 1 (the backward's dL/dscale leaves out its chain factor, as the reference does), and a
    precomputed covariance with scales and rotations absent (render() with pipe.compute_cov3D_python), including
    dL_dcov3D."""
    dev = cuda_device
    case = edge_scene(16, 3, seed=180)
    if source == "cov3D_precomp":
        cov = cov3d64(case["scales"], case["rotations"])
        fa, fwd, grads, bwd = run(case, dev, cov3D=cov)
        check_vs_oracle(case, fwd, grads, bwd, source, cov3D_precomp=cov)
        assert float(bwd[4].abs().max()) > 0.0
        assert float(bwd[6].abs().max()) == 0.0 and float(bwd[7].abs().max()) == 0.0  # no scales / rotations
    else:
        sm = float(source.split("_")[-1])
        fa, fwd, grads, bwd = run(case, dev, scale_modifier=sm)
        check_vs_oracle(case, fwd, grads, bwd, source, scale_modifier=sm)
    chain = ColourChain(case, fwd)
    chain.check_forward(source)
    chain.check_dsh(bwd[5], bwd[1], source)


# ------------------------------------------------------------------ projection edges
EDGES = ["fov_clamp", "near_plane", "flat", "quaternion_norm", "wide"]


def projection_scene(kind, seed):
    """edge_scene (M = 16, degree 3, 320 x 192) with one slot in three (those the scene leaves in front of the camera
    unless they fell in the off-screen tenth) moved to the edge under test."""
    case = edge_scene(16, 3, seed, W=320, H=192)
    cam = case["cam"]
    g = torch.Generator().manual_seed(seed + 11)
    sel = torch.arange(N) % 3 == 1
    n = int(sel.sum())
    u = lambda lo, hi, k=n: lo + (hi - lo) * torch.rand(k, generator=g, dtype=torch.float64)  # noqa: E731
    sign = torch.where(torch.rand(n, generator=g) < 0.5, -1.0, 1.0).double()
    lim_x, lim_y = 1.3 * cam.tanfovx, 1.3 * cam.tanfovy
    if kind == "fov_clamp":
        # view-space x/z (first half) or y/z (second half) within +-2 % of the Jacobian clamp at 1.3 tan(fov / 2);
        # splats large enough to reach into the image from there
        zv = u(3.0, 6.0)
        half = torch.arange(n) < n // 2
        xv = torch.where(half, sign * u(0.98, 1.02) * lim_x, u(-0.7, 0.7) * cam.tanfovx) * zv
        yv = torch.where(half, u(-0.7, 0.7) * cam.tanfovy, sign * u(0.98, 1.02) * lim_y) * zv
        case["means3D"][sel] = view_to_world(xv, yv, zv).float()
        case["scales"][sel] = torch.exp(torch.randn(n, 3, generator=g) * 0.2 + math.log(0.4))
    elif kind == "near_plane":
        zv = u(0.21, 0.3)  # just past the near plane at 0.2
        xv, yv = u(-0.9, 0.9) * cam.tanfovx * zv, u(-0.9, 0.9) * cam.tanfovy * zv
        case["means3D"][sel] = view_to_world(xv, yv, zv).float()
        case["scales"][sel] = torch.exp(torch.randn(n, 3, generator=g) * 0.3 + math.log(0.002))
    elif kind == "flat":
        # two scales near 1e-6: the projected footprint is a line, det_cov / det falls under the 2.5e-5 floor
        s = torch.empty(n, 3)
        s[:, 0] = torch.exp(torch.randn(n, generator=g) * 0.3 + math.log(0.05))
        s[:, 1:] = 1e-6 * (1.0 + 0.5 * torch.rand(n, 2, generator=g))
        case["scales"][sel] = s
        case["opacity"][sel] = 0.9 + 0.09 * torch.rand(n, 1, generator=g)
    elif kind == "quaternion_norm":
        # the rasterizer takes the quaternion as given (unnormalised), as the reference does
        case["rotations"][sel] *= u(0.3, 3.0).float()[:, None]
    elif kind == "wide":
        # every third selected slot a splat over more than 100 of the 20 x 12 tiles
        wide = torch.arange(N) % 9 == 1
        k = int(wide.sum())
        zv = u(3.0, 5.0, k)
        xv, yv = u(-0.5, 0.5, k) * cam.tanfovx * zv, u(-0.5, 0.5, k) * cam.tanfovy * zv
        case["means3D"][wide] = view_to_world(xv, yv, zv).float()
        case["scales"][wide] = torch.exp(torch.randn(k, 3, generator=g) * 0.1 + math.log(0.6))
    refresh_all_map(case)
    return case, sel


@pytest.mark.parametrize("kind", EDGES)
def test_projection_edges(cuda_device, kind):
    dev = cuda_device
    case, sel = projection_scene(kind, seed=200 + EDGES.index(kind))
    fa, fwd, grads, bwd = run(case, dev)
    live = (fwd[2] > 0).cpu()
    assert interleaved_rows(fwd) > 300, kind
    edge_live = live & sel
    assert int(edge_live.sum()) > 50, (kind, int(edge_live.sum()))
    so = check_vs_oracle(case, fwd, grads, bwd, kind)
    # the scene reaches the edge it is meant to test
    cam = case["cam"]
    m = case["means3D"].double()
    zv = m[:, 2] + 5.0
    if kind == "fov_clamp":
        rx, ry = (m[:, 0] / zv).abs() / (1.3 * cam.tanfovx), (m[:, 1] / zv).abs() / (1.3 * cam.tanfovy)
        beyond = edge_live & ((rx > 1.0) | (ry > 1.0))
        within = edge_live & (((rx > 0.98) & (rx < 1.0)) | ((ry > 0.98) & (ry < 1.0)))
        assert int(beyond.sum()) > 20 and int(within.sum()) > 20, (int(beyond.sum()), int(within.sum()))
    elif kind == "near_plane":
        assert float(zv[edge_live].min()) < 0.22 and float(zv[edge_live].max()) > 0.29
    elif kind == "flat":
        # opacity x h_scale at the floor sqrt(2.5e-5) in every visible flat slot
        h = torch.tensor(2.5e-5, dtype=torch.float32).sqrt()
        opac = so["records"].cpu()[:, 5][edge_live]
        assert torch.equal(opac, case["opacity"][:, 0][edge_live] * h)
    elif kind == "wide":
        assert int((so["tiles_touched"].cpu()[live] > 100).sum()) > 20
    chain = ColourChain(case, fwd)
    chain.check_forward(kind)
    chain.check_dsh(bwd[5], bwd[1], kind)
