"""PyTorch restatement of graphdeco 3DGS's adaptive density control (scene/gaussian_model.py of
graphdeco-inria/gaussian-splatting: densify_and_clone, densify_and_split, densification_postfix, prune_points,
_prune_optimizer, cat_tensors_to_optimizer, replace_tensor_to_optimizer, reset_opacity; utils/general_utils.py:
build_rotation, inverse_sigmoid) on separate parameter tensors and torch.optim.Adam state — the definition
hg_densify_plan / hg_densify_apply / hg_reset_opacity are held to (DESIGN.md §3 "Densify and prune").

Two departures, both part of this build's definition: the gradient statistic is the running maximum as accumulated
(not divided by the visit count), and the split draws can be injected (`samples`, the tensor torch.normal would
return) so that a test feeds the oracle and the kernel the same numbers.  Test infrastructure only."""
import torch

NAMES = ("xyz", "features", "opacity", "scaling", "rotation")


def inverse_sigmoid(x):
    return torch.log(x / (1 - x))


def build_rotation(r):
    norm = torch.sqrt(r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1] + r[:, 2] * r[:, 2] + r[:, 3] * r[:, 3])
    q = r / norm[:, None]
    R = torch.zeros((q.size(0), 3, 3), device=r.device)
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R[:, 0, 0] = 1 - 2 * (y * y + z * z)
    R[:, 0, 1] = 2 * (x * y - r * z)
    R[:, 0, 2] = 2 * (x * z + r * y)
    R[:, 1, 0] = 2 * (x * y + r * z)
    R[:, 1, 1] = 1 - 2 * (x * x + z * z)
    R[:, 1, 2] = 2 * (y * z - r * x)
    R[:, 2, 0] = 2 * (x * z - r * y)
    R[:, 2, 1] = 2 * (y * z + r * x)
    R[:, 2, 2] = 1 - 2 * (x * x + y * y)
    return R


class GaussianModel:
    """The parameter groups (raw: xyz, features [N,16,3], opacity logit, scaling log, rotation) in a torch.optim.Adam
    whose state holds the given moments and step count, and the three densification statistics."""

    def __init__(self, tensors, exp_avg, exp_avg_sq, step, accum, denom, max_radii2D, percent_dense=0.01):
        params = [torch.nn.Parameter(tensors[k].detach().clone().requires_grad_(True)) for k in NAMES]
        self.optimizer = torch.optim.Adam([{"params": [p], "lr": 0.0, "name": k} for k, p in zip(NAMES, params)],
                                          lr=0.0, eps=1e-15)
        for k, p in zip(NAMES, params):
            self.optimizer.state[p] = {"step": torch.tensor(float(step)), "exp_avg": exp_avg[k].detach().clone(),
                                       "exp_avg_sq": exp_avg_sq[k].detach().clone()}
        self._set(dict(zip(NAMES, params)))
        self.xyz_gradient_accum = accum.detach().clone().reshape(-1, 1)
        self.denom = denom.detach().clone().reshape(-1, 1)
        self.max_radii2D = max_radii2D.detach().clone().reshape(-1)
        self.percent_dense = percent_dense

    def _set(self, d):
        self._xyz, self._features, self._opacity = d["xyz"], d["features"], d["opacity"]
        self._scaling, self._rotation = d["scaling"], d["rotation"]

    get_xyz = property(lambda s: s._xyz)
    get_scaling = property(lambda s: torch.exp(s._scaling))
    get_opacity = property(lambda s: torch.sigmoid(s._opacity))

    def state(self, name):
        g = next(g for g in self.optimizer.param_groups if g["name"] == name)
        return self.optimizer.state[g["params"][0]]

    # ---- optimizer plumbing
    def replace_tensor_to_optimizer(self, tensor, name):
        optimizable_tensors = {}
        for group in self.optimizer.param_groups:
            if group["name"] == name:
                stored_state = self.optimizer.state.get(group["params"][0], None)
                stored_state["exp_avg"] = torch.zeros_like(tensor)
                stored_state["exp_avg_sq"] = torch.zeros_like(tensor)
                del self.optimizer.state[group["params"][0]]
                group["params"][0] = torch.nn.Parameter(tensor.requires_grad_(True))
                self.optimizer.state[group["params"][0]] = stored_state
                optimizable_tensors[group["name"]] = group["params"][0]
        return optimizable_tensors

    def _prune_optimizer(self, mask):
        optimizable_tensors = {}
        for group in self.optimizer.param_groups:
            stored_state = self.optimizer.state.get(group["params"][0], None)
            if stored_state is not None:
                stored_state["exp_avg"] = stored_state["exp_avg"][mask]
                stored_state["exp_avg_sq"] = stored_state["exp_avg_sq"][mask]
                del self.optimizer.state[group["params"][0]]
                group["params"][0] = torch.nn.Parameter((group["params"][0][mask].requires_grad_(True)))
                self.optimizer.state[group["params"][0]] = stored_state
            else:
                group["params"][0] = torch.nn.Parameter(group["params"][0][mask].requires_grad_(True))
            optimizable_tensors[group["name"]] = group["params"][0]
        return optimizable_tensors

    def prune_points(self, mask):
        valid_points_mask = ~mask
        self._set(self._prune_optimizer(valid_points_mask))
        self.xyz_gradient_accum = self.xyz_gradient_accum[valid_points_mask]
        self.denom = self.denom[valid_points_mask]
        self.max_radii2D = self.max_radii2D[valid_points_mask]

    def cat_tensors_to_optimizer(self, tensors_dict):
        optimizable_tensors = {}
        for group in self.optimizer.param_groups:
            extension_tensor = tensors_dict[group["name"]]
            stored_state = self.optimizer.state.get(group["params"][0], None)
            if stored_state is not None:
                stored_state["exp_avg"] = torch.cat((stored_state["exp_avg"], torch.zeros_like(extension_tensor)), dim=0)
                stored_state["exp_avg_sq"] = torch.cat((stored_state["exp_avg_sq"], torch.zeros_like(extension_tensor)),
                                                       dim=0)
                del self.optimizer.state[group["params"][0]]
                group["params"][0] = torch.nn.Parameter(torch.cat((group["params"][0], extension_tensor),
                                                                  dim=0).requires_grad_(True))
                self.optimizer.state[group["params"][0]] = stored_state
            else:
                group["params"][0] = torch.nn.Parameter(torch.cat((group["params"][0], extension_tensor),
                                                                  dim=0).requires_grad_(True))
            optimizable_tensors[group["name"]] = group["params"][0]
        return optimizable_tensors

    def densification_postfix(self, new_xyz, new_features, new_opacities, new_scaling, new_rotation):
        d = {"xyz": new_xyz, "features": new_features, "opacity": new_opacities, "scaling": new_scaling,
             "rotation": new_rotation}
        self._set(self.cat_tensors_to_optimizer(d))
        dev = self._xyz.device
        self.xyz_gradient_accum = torch.zeros((self._xyz.shape[0], 1), device=dev)
        self.denom = torch.zeros((self._xyz.shape[0], 1), device=dev)
        self.max_radii2D = torch.zeros((self._xyz.shape[0]), device=dev)

    # ---- adaptive density control
    def densify_and_split(self, grads, grad_threshold, scene_extent, N=2, samples=None):
        n_init_points = self._xyz.shape[0]
        padded_grad = torch.zeros((n_init_points), device=self._xyz.device)
        padded_grad[:grads.shape[0]] = grads.squeeze()
        selected_pts_mask = torch.where(padded_grad >= grad_threshold, True, False)
        selected_pts_mask = torch.logical_and(selected_pts_mask,
                                              torch.max(self.get_scaling, dim=1).values > self.percent_dense * scene_extent)
        self.n_split = int(selected_pts_mask.sum())
        stds = self.get_scaling[selected_pts_mask].repeat(N, 1)
        if samples is None:
            means = torch.zeros((stds.size(0), 3), device=self._xyz.device)
            samples = torch.normal(mean=means, std=stds)
        rots = build_rotation(self._rotation[selected_pts_mask]).repeat(N, 1, 1)
        new_xyz = torch.bmm(rots, samples.unsqueeze(-1)).squeeze(-1) + self.get_xyz[selected_pts_mask].repeat(N, 1)
        new_scaling = torch.log(self.get_scaling[selected_pts_mask].repeat(N, 1) / (0.8 * N))
        new_rotation = self._rotation[selected_pts_mask].repeat(N, 1)
        new_features = self._features[selected_pts_mask].repeat(N, 1, 1)
        new_opacity = self._opacity[selected_pts_mask].repeat(N, 1)
        self.densification_postfix(new_xyz, new_features, new_opacity, new_scaling, new_rotation)
        prune_filter = torch.cat((selected_pts_mask, torch.zeros(N * selected_pts_mask.sum(), device=self._xyz.device,
                                                                 dtype=bool)))
        self.prune_points(prune_filter)

    def densify_and_clone(self, grads, grad_threshold, scene_extent):
        selected_pts_mask = torch.where(torch.norm(grads, dim=-1) >= grad_threshold, True, False)
        selected_pts_mask = torch.logical_and(selected_pts_mask,
                                              torch.max(self.get_scaling, dim=1).values <= self.percent_dense * scene_extent)
        self.densification_postfix(self._xyz[selected_pts_mask], self._features[selected_pts_mask],
                                   self._opacity[selected_pts_mask], self._scaling[selected_pts_mask],
                                   self._rotation[selected_pts_mask])

    def densify_and_prune(self, max_grad, min_opacity, extent, max_screen_size, samples=None):
        grads = self.xyz_gradient_accum.clone()  # this build: the running maximum as accumulated, not / denom
        grads[grads.isnan()] = 0.0
        self.densify_and_clone(grads, max_grad, extent)
        n_before = self._xyz.shape[0]
        self.densify_and_split(grads, max_grad, extent, samples=samples)
        first_child = n_before - int(self.n_split)
        prune_mask = (self.get_opacity < min_opacity).squeeze(1)  # (squeeze(): a 0-dim mask at one row)
        if max_screen_size:
            big_points_vs = self.max_radii2D > max_screen_size  # zero after densification_postfix: never true
            big_points_ws = self.get_scaling.max(dim=1).values > 0.1 * extent
            prune_mask = torch.logical_or(torch.logical_or(prune_mask, big_points_vs), big_points_ws)
        self.prune_points(prune_mask)
        # (for tests) rows of the result that are children: [first_child_row, end); the split draws they were made from
        self.first_child_row = first_child - int(prune_mask[:first_child].sum())
        self.kept_children = ~prune_mask[first_child:]

    def reset_opacity(self):
        opacities_new = inverse_sigmoid(torch.min(self.get_opacity, torch.ones_like(self.get_opacity) * 0.01))
        self._opacity = self.replace_tensor_to_optimizer(opacities_new, "opacity")["opacity"]
