"""GPU parity tests of the hand-written binning stage (hidegs_b200/csrc/binning.cu): tile buckets + per-tile
shared-memory radix sort against the reference's global 64-bit key sort (rasterizer_impl.cu:321-371).

Bit-exact bar: num_rendered, the sorted 64-bit keys, point_list and the tile ranges — including equal depths
(the reference's stable sort leaves them in ascending slot order) and lists of every length class the sort
dispatches on (one warp <= 1024 — packed one-word elements, with the general routine as its fallback —, one CTA <= 2048,
512-thread CTA <= 12288, HBM scratch beyond).  At every one of them the blend that walks those lists is held to the CPU
oracle too: colour, contributor counts, final transmittance and observe counts of the forward, and the gradients of the
backward."""
import numpy as np
import pytest
import torch

import raster_utils as ru

pytestmark = pytest.mark.gpu


def _forward(case, dev):
    fa = ru.op_args(case, dev)
    fwd = ru.OUR_C.rasterize_gaussians(*fa)
    torch.cuda.synchronize()
    return fa, fwd


def _check(case, dev, what, min_longest=0, max_longest=None):
    fa, ours = _forward(case, dev)
    so = ru.our_state(ours, case["P"], case["W"], case["H"])
    o = ru.oracle_for_case(case)
    oo = o.forward()
    assert ours[0] == oo["num_rendered"] and ours[0] > 0, what
    rng = oo["ranges"].reshape(-1, 2).astype(np.int64)
    longest = int((rng[:, 1] - rng[:, 0]).max())
    assert longest >= min_longest, "%s: longest list %d does not reach the class under test" % (what, longest)
    if max_longest is not None:
        assert longest <= max_longest, "%s: longest list %d leaves the class under test" % (what, longest)
    assert np.array_equal(so["keys"].cpu().numpy().view(np.uint64), oo["keys"]), what + ": sorted keys"
    assert np.array_equal(so["point_list"].cpu().numpy().view(np.uint32), oo["point_list"]), what + ": point_list"
    assert np.array_equal(so["ranges"].cpu().numpy().view(np.uint32), oo["ranges"]), what + ": ranges"
    assert np.array_equal(so["keys_unsorted"].cpu().numpy().view(np.uint64), oo["keys_unsorted"]), what + ": emission"
    # the blend over these lists: the forward's images and per-pixel state (the oracle's expf is the C library's, within
    # 2 ulp of the GPU's: pixel values agree to ~1e-6, alpha decisions and so contributor counts exactly) ...
    img = lambda t: torch.as_tensor(t).double().cpu()  # noqa: E731
    for name, a, b in (("colour", ours[1], oo["color"]), ("all_map", ours[4], oo["all_map"]),
                       ("final_T", so["final_T"], oo["final_T"])):
        err = float((img(a) - img(b)).abs().max())
        assert err <= 1e-4, "%s: %s off by %.3g" % (what, name, err)
    assert np.array_equal(so["n_contrib"].cpu().numpy().view(np.uint32), oo["n_contrib"]), what + ": n_contrib"
    assert np.array_equal(ours[3].cpu().numpy(), oo["out_observe"]), what + ": out_observe"
    # ... and the backward's gradients
    grads = ru.syn.upstream_grads(case["W"], case["H"])
    ours_b = ru.OUR_C.rasterize_gaussians_backward(*ru.bwd_args(fa, ours, grads, dev))
    og = o.backward(grads["color"].numpy(), grads["all_map"].numpy(), grads["plane_depth"].numpy(),
                    grads["invdepth"].numpy())
    ru.assert_grads_close([g.cpu() for g in ours_b], [torch.from_numpy(og[n]) for n in ru.GRAD_NAMES], what=what)
    if ru.ref_available():
        ref = ru.ref_module().rasterize_gaussians(*fa)
        torch.cuda.synchronize()
        sr = ru.ref_state(ref, case["P"], case["W"], case["H"])
        assert ours[0] == ref[0]
        for k in ("keys", "point_list", "ranges", "n_contrib"):
            assert torch.equal(so[k], sr[k]), "%s vs reference: %s" % (what, k)
    return longest


def _duplicate_rows(case, rows, copies, seed):
    """Append `copies` exact copies of the given Gaussians at random positions (identical depth in every tile)."""
    g = torch.Generator().manual_seed(seed)
    n = case["means3D"].shape[0]
    src = torch.cat([torch.arange(n), rows.repeat(copies)])
    src = src[torch.randperm(src.numel(), generator=g)]
    for k in ("means3D", "scales", "rotations", "opacity", "shs", "all_map"):
        case[k] = case[k][src].contiguous()
    case["P"] = src.numel()
    return case


def test_equal_depths_short_runs(cuda_device):
    case = ru.build_case(5000, 208, 120, seed=31)
    g = torch.Generator().manual_seed(5)
    rows = torch.randperm(5000, generator=g)[:600]
    case = _duplicate_rows(case, rows, 3, seed=6)  # runs of 4 equal keys
    _check(case, cuda_device, "short runs")


def test_equal_depths_long_runs(cuda_device):
    case = ru.build_case(3000, 208, 120, seed=32)
    g = torch.Generator().manual_seed(7)
    rows = torch.randperm(3000, generator=g)[:20]
    case = _duplicate_rows(case, rows, 60, seed=8)  # runs of 61 equal keys: the slot-first re-sort
    _check(case, cuda_device, "long runs")


def test_all_depths_equal(cuda_device):
    """A fronto-parallel sheet of splats: every key of a list is the same, the order is the slot order alone."""
    case = ru.build_case(6000, 208, 120, seed=33)
    case["means3D"][:, 2] = 0.25
    case["all_map"] = ru.syn.geometry_all_map(case["means3D"], case["scales"], case["rotations"], case["cam"])
    fa, ours = _forward(case, cuda_device)
    so = ru.our_state(ours, case["P"], case["W"], case["H"])
    d = so["depths"][ours[2] > 0]
    assert d.numel() > 1000 and float(d.max() - d.min()) == 0.0  # the premise of the test
    _check(case, cuda_device, "sheet")


@pytest.mark.parametrize("what,n,scale,lo,hi", [
    ("medium and long lists", 6000, 0.35, 1025, 4096),       # lists of 1892 .. 3720: CTA (<= 2048) and 512-thread CTA
    ("long lists (512-thread CTA)", 12000, 0.6, 4097, 12288),  # 6368 .. 10061
    ("lists beyond shared memory", 30000, 1.2, 12289, None),   # 25850 .. 29432
])
def test_list_length_classes(cuda_device, what, n, scale, lo, hi):
    import math
    case = ru.build_case(n, 64, 48, seed=41, log_scale_mean=math.log(scale))
    _check(case, cuda_device, what, min_longest=lo, max_longest=hi)


def test_lists_beyond_shared_memory_low_opacity(cuda_device):
    """The longest class at opacity 0.02: the transmittance falls slowly, so each pixel's walk goes on for 1079 .. 1732
    entries (9 .. 14 of the forward's 128-entry batches, up to ~100 of the backward's 16-entry MMA groups) instead of
    the 24 .. 46 of the default opacities (measured with the oracle)."""
    import math
    case = ru.build_case(30000, 64, 48, seed=41, log_scale_mean=math.log(1.2))
    case["opacity"] = torch.full_like(case["opacity"], 0.02)
    _check(case, cuda_device, "lists beyond shared memory, opacity 0.02", min_longest=12289)


def test_wide_depth_range_short_lists(cuda_device):
    """Depths from 0.3 to 2e5 inside one tile: more than 27 significant key bits, so lists of 513..1024 entries do not
    fit the one-word packing of the short-list path and take its fallback (67 such lists in this scene)."""
    import math
    n = 3000
    case = ru.build_case(n, 208, 120, seed=51, log_scale_mean=math.log(0.06))
    g = torch.Generator().manual_seed(3)
    z = torch.exp(torch.rand(n, generator=g) * (math.log(2e5) - math.log(0.3)) + math.log(0.3))
    xy = (torch.rand(n, 2, generator=g) * 2 - 1) * torch.tensor([0.55, 0.3])
    case["means3D"] = torch.cat([xy * z[:, None], (z - 5.0)[:, None]], 1).contiguous()
    case["scales"] = (case["scales"] * z[:, None]).contiguous()
    case["all_map"] = ru.syn.geometry_all_map(case["means3D"], case["scales"], case["rotations"], case["cam"])
    _check(case, cuda_device, "wide depth range", min_longest=513)


def test_mixed_classes_with_ties(cuda_device):
    """Long lists AND equal depths: the slot-first re-sort in the multi-warp and the HBM-scratch variants."""
    import math
    case = ru.build_case(9000, 64, 48, seed=42, log_scale_mean=math.log(1.0))
    g = torch.Generator().manual_seed(9)
    rows = torch.randperm(9000, generator=g)[:40]
    case = _duplicate_rows(case, rows, 100, seed=10)
    _check(case, cuda_device, "mixed", min_longest=4097)
