"""Helpers shared by the rasterizer parity tests (not collected by pytest)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

from hidegs_b200 import _lib, synthetic as syn  # noqa: E402
from hidegs_b200.diff_gaussian_rasterization import _C as OUR_C  # noqa: E402


# --------------------------------------------------------------------- scenes
def build_case(n, W, H, seed=0, log_scale_mean=None, device="cpu", sh_degree=3, with_hier=False,
               with_indices=False, eye=(0.0, 0.0, -5.0), sh_coeffs=16):
    """Synthetic scene + camera + all_map (+ optional hierarchy inputs), CPU tensors."""
    import math
    cam = syn.default_camera(W, H, eye=eye)
    if log_scale_mean is None:
        # keep the splat footprint in pixels similar to config 2 (sigma ~ 3 px at 1080p)
        log_scale_mean = math.log(0.01 * 1920.0 / W)
    sc = syn.make_scene(n, seed=seed, log_scale_mean=log_scale_mean, sh_coeffs=sh_coeffs)
    g = torch.Generator().manual_seed(seed + 1000)
    case = dict(cam=cam, W=W, H=H, sh_degree=sh_degree, **sc)
    P = n
    if with_indices:
        perm = torch.randperm(n, generator=g)[: max(1, (n * 3) // 5)].sort()[0].to(torch.int32)
        case["render_indices"] = perm
        P = perm.numel()
        # Parents come from the NON-rendered rows, as in a hierarchy cut (a node and its parent are
        # never rendered together; otherwise the reference's parent push races with the parent's own
        # gradient write, backward.cu:449,485-488).
        rest = torch.ones(n, dtype=torch.bool)
        rest[perm.long()] = False
        rest = rest.nonzero().flatten()
        case["parent_indices"] = rest[torch.randint(0, rest.numel(), (P,), generator=g)].to(torch.int32)
        case["parent_indices"][::7] = -1
    if with_hier:
        ts = torch.rand(P, generator=g)
        ts[torch.rand(P, generator=g) < 0.5] = 1.0
        case["interpolation_weights"] = ts
        case["num_node_kids"] = torch.randint(2, 9, (P,), generator=g, dtype=torch.int32)
    src = case["render_indices"].long() if with_indices else slice(None)
    case["all_map"] = syn.geometry_all_map(sc["means3D"][src], sc["scales"][src], sc["rotations"][src], cam)
    case["P"] = P
    return case


def op_args(case, device, render_geo=True, do_depth=True, bg=(0.1, 0.2, 0.3), colors_precomp=None):
    """Positional argument tuple of `_C.rasterize_gaussians` for a case."""
    cam = case["cam"]
    e_i = torch.empty(0, dtype=torch.int32, device=device)
    e_f = torch.empty(0, dtype=torch.float32, device=device)
    d = lambda k, e: case[k].to(device) if k in case else e  # noqa: E731
    use_sh = colors_precomp is None
    return (torch.tensor(bg, dtype=torch.float32, device=device), d("render_indices", e_i), d("parent_indices", e_i),
            d("interpolation_weights", e_f), d("num_node_kids", e_i), case["means3D"].to(device),
            e_f if use_sh else colors_precomp.to(device), case["all_map"].to(device), case["opacity"].to(device),
            case["scales"].to(device), case["rotations"].to(device), 1.0, e_f,
            cam.world_view_transform.to(device), cam.full_proj_transform.to(device), cam.tanfovx, cam.tanfovy,
            case["H"], case["W"], case["shs"].to(device) if use_sh else e_f, case["sh_degree"],
            cam.camera_center.to(device), False, render_geo, False, do_depth)


def bwd_args(fargs, fwd_out, grads, device):
    """Positional argument tuple of `_C.rasterize_gaussians_backward`."""
    (bg, indices, parents, ts, kids, means3D, colors, all_map, opacity, scales, rotations, scale_modifier, cov3D,
     view, proj, tfx, tfy, H, W, sh, degree, campos, prefiltered, render_geo, debug, do_depth) = fargs
    R, color, radii, observe, out_all_map, plane_depth, geom, binning, img, invdepth = fwd_out
    return (bg, out_all_map, indices, parents, ts, kids, means3D, radii, colors, all_map, opacity, scales, rotations,
            scale_modifier, cov3D, view, proj, tfx, tfy, grads["color"].to(device), grads["all_map"].to(device),
            grads["plane_depth"].to(device), grads["invdepth"].to(device), sh, degree, campos, geom, R, binning, img,
            render_geo, debug)


GRAD_NAMES = ("dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dscales",
              "dL_drotations", "dL_dall_map")


# --------------------------------------------------------- our state accessors
def our_state(fwd_out, P, W, H):
    """Slice our opaque buffers into named tensors (keys, sorted list, ranges, ...)."""
    R, color, radii, observe, all_map, plane_depth, geom, binning, img, invdepth = fwd_out
    L = _lib.layout(P, W, H, R)

    def base(t):
        off = (-t.data_ptr()) % 256
        return t[off:]

    def view(buf, off, nbytes, dtype):
        return base(buf)[off:off + nbytes].view(dtype)

    T = ((W + 15) // 16) * ((H + 15) // 16)
    st = dict(R=R)
    st["depths"] = view(geom, L.depths, 4 * P, torch.float32)
    st["tiles_touched"] = view(geom, L.tiles_touched, 4 * P, torch.int32)
    st["rects"] = view(geom, L.rects, 8 * P, torch.int32).view(P, 2)
    st["cov3D"] = view(geom, L.cov3D, 24 * P, torch.float32).view(P, 6)
    st["clamped"] = view(geom, L.clamped, P, torch.uint8)
    st["records"] = view(geom, L.records, 64 * P, torch.float32).view(P, 16)
    st["final_T"] = view(img, L.final_T, 4 * W * H, torch.float32)
    st["n_contrib"] = view(img, L.n_contrib, 4 * W * H, torch.int32)
    st["ranges"] = view(img, L.ranges, 8 * T, torch.int32).view(T, 2)
    if R > 0:
        st["point_list"] = view(binning, L.vals, 4 * R, torch.int32)
        # The library buckets the instances by tile and sorts each list on chip; it never holds the reference's 64-bit
        # tile|depth keys.  hg_raster_debug_keys rebuilds them from its buffers (see include/hidegs_raster.h).
        dev = geom.device
        st["keys_unsorted"] = torch.empty(R, dtype=torch.int64, device=dev)
        st["vals_unsorted"] = torch.empty(R, dtype=torch.int32, device=dev)
        st["keys"] = torch.empty(R, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            rc = _lib.lib().hg_raster_debug_keys(P, W, H, R, radii.data_ptr(), geom.data_ptr(), binning.data_ptr(),
                                                 st["keys_unsorted"].data_ptr(), st["vals_unsorted"].data_ptr(),
                                                 st["keys"].data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "hg_raster_debug_keys")
        torch.cuda.synchronize(dev)
    return st


# ------------------------------------------------------------ reference (_ref)
_ref_mod = None


def ref_available():
    return os.path.exists(os.path.join(REF_DIR, "ref_rasterizer_C.so"))


def ref_module():
    """The UNMODIFIED reference rasterizer built for sm_100 by oracle/Makefile (`make ref`)."""
    global _ref_mod
    if _ref_mod is None:
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import ref_rasterizer_C  # noqa: E402
        _ref_mod = ref_rasterizer_C
    return _ref_mod


def _align128(x):
    return (x + 127) & ~127


def ref_state(fwd_out, P, W, H):
    """Parse the reference's three byte buffers (GeometryState/ImageState/BinningState::fromChunk,
    rasterizer_impl.cu:159-199: every array aligned to 128 B on the absolute address)."""
    R, color, radii, observe, all_map, plane_depth, geom, binning, img, invdepth = fwd_out
    st = dict(R=R)

    def carve(buf, specs):
        out = {}
        addr = buf.data_ptr()
        cur = addr
        for name, nbytes, dtype in specs:
            cur = _align128(cur)
            out[name] = buf[cur - addr: cur - addr + nbytes].view(dtype)
            cur += nbytes
        return out

    g = carve(geom, [("depths", 4 * P, torch.float32), ("clamped", 3 * P, torch.uint8), ("p_clamped", 3 * P, torch.uint8),
                     ("internal_radii", 4 * P, torch.int32), ("means2D", 8 * P, torch.float32),
                     ("cov3D", 24 * P, torch.float32), ("conic_opacity", 16 * P, torch.float32),
                     ("rgb", 12 * P, torch.float32), ("tiles_touched", 4 * P, torch.int32)])
    st.update(g)
    st["means2D"] = st["means2D"].view(P, 2)
    st["cov3D"] = st["cov3D"].view(P, 6)
    st["conic_opacity"] = st["conic_opacity"].view(P, 4)
    st["rgb"] = st["rgb"].view(P, 3)
    st["clamped"] = st["clamped"].view(P, 3)
    HW = W * H
    i = carve(img, [("final_T", 4 * HW, torch.float32), ("n_contrib", 4 * HW, torch.int32), ("ranges", 8 * HW, torch.int32)])
    T = ((W + 15) // 16) * ((H + 15) // 16)
    st["final_T"], st["n_contrib"] = i["final_T"], i["n_contrib"]
    st["ranges"] = i["ranges"].view(HW, 2)[:T]
    if R > 0:
        b = carve(binning, [("point_list", 4 * R, torch.int32), ("vals_unsorted", 4 * R, torch.int32),
                            ("keys", 8 * R, torch.int64), ("keys_unsorted", 8 * R, torch.int64)])
        st.update(b)
    return st


def mask_undefined_parent_rows(case, named_grads):
    """Drop the rows of dL_dmeans3D whose value is undefined in the reference.

    For a slot with a parent the reference's forward records the SH clamp flags in `p_clamped`
    (forward.cu:411) but its backward reads `clamped` (backward.cu:453), which that path never
    wrote: the view-direction part of the child's mean gradient -- pushed to the PARENT row,
    backward.cu:485-488 -- depends on whatever bytes the allocator recycled (verified on the B200:
    the reference's value equals the oracle's with all three flags forced on for some children and
    off for others).  hidegs_b200 and the oracle define those flags as "not clamped".  With SH
    degree 0 the direction term vanishes and every row is comparable."""
    if "parent_indices" not in case or case["sh_degree"] == 0:
        return named_grads
    par = case["parent_indices"].long()
    rows = torch.unique(par[par >= 0])
    out = dict(named_grads)
    g = out["dL_dmeans3D"].detach().cpu().clone()
    g[rows] = 0.0
    out["dL_dmeans3D"] = g
    return out


# ----------------------------------------------------------------- comparisons
def rel_report(a, b):
    """(max abs err, max |b|, fraction of elements outside rtol 1e-3 / atol 1e-5*max|b|)."""
    a, b = a.double().flatten(), b.double().flatten()
    if a.numel() == 0:
        return 0.0, 0.0, 0.0
    err = (a - b).abs()
    scale = float(b.abs().max())
    tol = 1e-3 * b.abs() + 1e-5 * max(scale, 1e-30)
    return float(err.max()), scale, float((err > tol).double().mean())


# Element-wise floor per gradient tensor, as a fraction of rtol * max|b|.  A floor is needed where an entry is the
# (float-atomic-order dependent) sum of terms much larger than itself:
#   dL_dcov3D / dL_dscales / dL_drotations  chain dL/dconic through T^2 and the covariance factorisation: 3e-2
#   dL_dmeans3D                              sums the projection, covariance and SH-direction paths, which cancel: 3e-2
#   everything else (colours, opacity, 2-D means, SH rows, geometry channels) is a plain per-pixel sum: 1e-2
FLOOR_BY_TENSOR = {"dL_dcov3D": 3e-2, "dL_dscales": 3e-2, "dL_drotations": 3e-2, "dL_dmeans3D": 3e-2,
                   # the same three groups under the trainer's parameter names (raw parameters: + the activation chain)
                   "xyz": 3e-2, "scaling": 3e-2, "rotation": 3e-2}
DEFAULT_FLOOR = 1e-2


def assert_grads_close(ours, theirs, names=GRAD_NAMES, rtol=1e-3, floor=None, l2_tol=1e-4, what="", max_bad_frac=0.0):
    """Gradients within `rtol` relative.  Two criteria per tensor:
      * relative L2 error  ||a-b|| / ||b||  <= l2_tol, and
      * element-wise |a-b| <= rtol*|b| + rtol*floor*max|b|  (the floor absorbs summation-order noise on
        entries that are small next to the terms that cancel into them; per tensor, FLOOR_BY_TENSOR, unless `floor`
        is given).
    `max_bad_frac`: fraction of elements allowed outside the element-wise bound (0 except for the multi-million
    element full-size cases, where single cancellation-dominated entries of both implementations are atomic-order noise).
    """
    for name, a, b in zip(names, ours, theirs):
        a, b = torch.as_tensor(a).detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
        assert a.shape == b.shape, (name, a.shape, b.shape)
        if a.numel() == 0:
            continue
        scale = float(b.abs().max())
        l2 = float((a - b).norm()) / max(float(b.norm()), 1e-30)
        assert l2 <= l2_tol or scale == 0.0, "%s %s: relative L2 error %.3g" % (what, name, l2)
        fl = floor if floor is not None else FLOOR_BY_TENSOR.get(name, DEFAULT_FLOOR)
        tol = rtol * b.abs() + rtol * fl * scale + 1e-30
        bad = (a - b).abs() > tol
        frac = float(bad.double().mean())
        assert frac <= max_bad_frac, "%s %s: %.3g%% of elements off (max err %.3g, scale %.3g)" % (
            what, name, 100 * frac, float((a - b).abs().max()), scale)


def oracle_for_case(case, render_geo=True, do_depth=True, bg=(0.1, 0.2, 0.3), colors_precomp=None, nthreads=1,
                    scale_modifier=1.0, cov3D_precomp=None):
    """CPU oracle (oracle/raster_oracle.py) configured like op_args().  With `cov3D_precomp` the scales and rotations
    are left out, as render() does when it precomputes the covariance."""
    from oracle.raster_oracle import OracleRasterizer
    cam = case["cam"]
    n = lambda k: case[k].numpy() if k in case else None  # noqa: E731
    return OracleRasterizer(
        bg=np.array(bg, np.float32), viewmatrix=cam.world_view_transform.numpy(),
        projmatrix=cam.full_proj_transform.numpy(), campos=cam.camera_center.numpy(), means3D=case["means3D"].numpy(),
        opacities=case["opacity"].numpy(), image_height=case["H"], image_width=case["W"], tanfovx=cam.tanfovx,
        tanfovy=cam.tanfovy, shs=case["shs"].numpy() if colors_precomp is None else None,
        colors_precomp=None if colors_precomp is None else colors_precomp.numpy(), all_map=case["all_map"].numpy(),
        scales=None if cov3D_precomp is not None else case["scales"].numpy(),
        rotations=None if cov3D_precomp is not None else case["rotations"].numpy(),
        cov3D_precomp=None if cov3D_precomp is None else cov3D_precomp.numpy(), scale_modifier=scale_modifier,
        sh_degree=case["sh_degree"],
        render_indices=n("render_indices"), parent_indices=n("parent_indices"),
        interpolation_weights=n("interpolation_weights"), num_node_kids=n("num_node_kids"), render_geo=render_geo,
        do_depth=do_depth, nthreads=nthreads)
