"""PyTorch restatement of 3DGS-MCMC densification (Kheradmand et al., 2024; gsplat's MCMCStrategy: relocate,
sample_add, compute_relocation, inject_noise_to_position) over separate parameter tensors, in float64 where the
definition evaluates in double — the definition hg_mcmc_regularizer / hg_mcmc_inject_noise / hg_mcmc_relocate /
hg_mcmc_grow are held to (DESIGN.md §3 "MCMC densification").  The formulas are the paper's and gsplat's as recalled,
not checked against a reference tree.

Departures from gsplat, all part of this build's definition: the relocation formula is evaluated in float64 and rounded
once (gsplat: float32); relocation zeroes the moments of the destinations as well as of the sources; growth zeroes the
moments of the sources.  The draws are injected (`sources`, the rows torch.multinomial would return) so that a test
feeds the oracle and the kernels the same numbers.  Test infrastructure only."""
import math

import torch

NAMES = ("xyz", "features", "opacity", "scaling", "rotation")
N_MAX = 51
FLT_EPSILON = 2.0 ** -23


def build_rotation(r):
    """graphdeco's build_rotation in the dtype of r."""
    q = r / torch.sqrt((r * r).sum(dim=1, keepdim=True))
    w, x, y, z = q.unbind(1)
    return torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                        2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                        2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], dim=1).view(-1, 3, 3)


def relocation(o, s, n, min_opacity=None):
    """compute_relocation in float64: o' = 1 - (1 - o)^(1/n), s' = s o / sum_{i=1..n} sum_{k=0..i-1} C(i-1, k) (-1)^k
    / sqrt(k+1) o'^(k+1), with n clamped to [1, 51]; o' then clamped to [min_opacity, 1 - FLT_EPSILON] unless
    min_opacity is None.  o [M], s [M, 3], n [M] integers; returns (o', s') as float64."""
    o = torch.as_tensor(o, dtype=torch.float64)
    s = torch.as_tensor(s, dtype=torch.float64)
    n = torch.as_tensor(n).to(torch.int64).clamp(1, N_MAX)
    op = 1.0 - torch.pow(1.0 - o, 1.0 / n.to(torch.float64))
    denom = torch.zeros_like(o)
    for i in range(1, N_MAX + 1):
        inner = torch.zeros_like(o)
        for k in range(i):
            inner = inner + math.comb(i - 1, k) * (-1.0) ** k / math.sqrt(k + 1) * op ** (k + 1)
        denom = torch.where(n >= i, denom + inner, denom)
    s2 = s * o[:, None] / denom[:, None]
    if min_opacity is not None:
        op = op.clamp(float(min_opacity), 1.0 - FLT_EPSILON)
    return op, s2


def activated_opacity(opacity_logit):
    """o in float32 with the kernels' bits (1 / (1 + exp(-x)), as activate_kernel and torch.sigmoid)."""
    return 1.0 / (1.0 + torch.exp(-opacity_logit.float()))


def relocated_raw(opacity_logit, scaling_log, counts, min_opacity):
    """(logit(o'), log(s')) rounded once to float32 for rows drawn `counts` >= 1 times (n = counts + 1)."""
    o = activated_opacity(opacity_logit).reshape(-1).double()
    s = torch.exp(scaling_log.float()).double().reshape(-1, 3)
    op, s2 = relocation(o, s, counts + 1, min_opacity)
    return torch.log(op / (1.0 - op)).float(), torch.log(s2).float()


def regularizer(opacity_logit, scaling_log, opacity_reg, scale_reg):
    """(Reg, dReg/dopacity_logit, dReg/dscaling_log) in float64 autograd."""
    x = opacity_logit.detach().double().requires_grad_(True)
    y = scaling_log.detach().double().requires_grad_(True)
    reg = opacity_reg * torch.sigmoid(x).mean() + scale_reg * torch.exp(y).mean()
    reg.backward()
    return reg.detach(), x.grad, y.grad


def noise_delta(opacity_logit, scaling_log, rotation, z, scale):
    """inject_noise_to_position's increment: scale sigma(100 ((1 - o) - 0.995)) (R diag(s^2) R^T) z, the gate in
    float32 as gsplat evaluates it (its argument multiplies the rounding of 1 - o and of 0.995 by 100, which a float64
    gate would count as a 1e-5 error of the kernel), everything after it in float64."""
    o = activated_opacity(opacity_logit).reshape(-1)
    gate = (1.0 / (1.0 + torch.exp(-100.0 * ((1.0 - o) - 0.995)))).double()
    R = build_rotation(rotation.double())
    s2 = torch.exp(scaling_log.double()) ** 2
    cov = R @ torch.diag_embed(s2) @ R.transpose(1, 2)
    v = z.double() * gate[:, None] * float(scale)
    return (cov @ v.unsqueeze(-1)).squeeze(-1)


def _counts(sources, N):
    return torch.bincount(sources, minlength=N)


def relocate(t, m, v, sources, min_opacity):
    """Relocation over dicts of float32 tensors {name: [N, ...]} (parameters and both moments, on one device; on the
    kernels' device the activations have their bits): dead rows
    (sigmoid(opacity) <= min_opacity, NaN included) in row order take sources[j]; returns new dicts."""
    t, m, v = ({k: x.detach().clone() for k, x in d.items()} for d in (t, m, v))
    N = t["xyz"].shape[0]
    sources = torch.as_tensor(sources).to(t["xyz"].device).long()
    dead = (~(activated_opacity(t["opacity"]).reshape(-1) > min_opacity)).nonzero().view(-1)
    alive = int(N - dead.numel())
    if dead.numel() == 0 or alive == 0:
        return t, m, v
    sources = sources[:dead.numel()]
    c = _counts(sources, N)
    drawn = (c > 0).nonzero().view(-1)
    nl, ns = relocated_raw(t["opacity"][drawn], t["scaling"][drawn], c[drawn], min_opacity)
    t["opacity"][drawn] = nl.view(-1, 1)
    t["scaling"][drawn] = ns
    for k in NAMES:
        t[k][dead[:sources.numel()]] = t[k][sources]
        for mom in (m, v):
            mom[k][drawn] = 0.0
            mom[k][dead[:sources.numel()]] = 0.0
    return t, m, v


def grow(t, m, v, sources, min_opacity):
    """Growth by len(sources) rows: the sources take (o', s') and zero moments, their copies are appended in draw order
    with zero moments; returns new dicts."""
    t, m, v = ({k: x.detach().clone() for k, x in d.items()} for d in (t, m, v))
    N = t["xyz"].shape[0]
    sources = torch.as_tensor(sources).to(t["xyz"].device).long()
    c = _counts(sources, N)
    drawn = (c > 0).nonzero().view(-1)
    nl, ns = relocated_raw(t["opacity"][drawn], t["scaling"][drawn], c[drawn], min_opacity)
    t["opacity"][drawn] = nl.view(-1, 1)
    t["scaling"][drawn] = ns
    for k in NAMES:
        t[k] = torch.cat([t[k], t[k][sources]])
        for mom in (m, v):
            mom[k][drawn] = 0.0
            mom[k] = torch.cat([mom[k], torch.zeros_like(mom[k][sources])])
    return t, m, v
