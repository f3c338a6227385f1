"""point_cloud.ply / point_cloud.bin of a Gaussian model (SURVEY.md §8(f) f4), the on-disk formats the reference reads and
writes around training: `GaussianModel.save_ply` (scene/gaussian_model.py:526-544), `load_ply_file` / `load_ply`
(:322-355, :548-558), `construct_list_of_attributes` (:472-484), and the raw dump at the end of `save_pt` (:507-517).

The reference goes through `plyfile` (PlyData / PlyElement, requirements.txt:158 plyfile==1.1): it builds one tuple per
Gaussian on the host (`list(map(tuple, attributes))`) and lets plyfile emit a binary little-endian `vertex` element of
62 float properties.  Here the 62-column row matrix is assembled where the tensors live (one `torch.cat` on the GPU for
CUDA tensors), crosses to the host once, and is written with one `tofile`; reading parses the header, maps the file and
splits the columns by NAME (any property order, extra float properties ignored), exactly the fields the reference reads.
"""
import json
import os
import struct

import numpy as np
import torch

_PLY_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "<i2", "int16": "<i2", "ushort": "<u2",
              "uint16": "<u2", "int": "<i4", "int32": "<i4", "uint": "<u4", "uint32": "<u4", "float": "<f4",
              "float32": "<f4", "double": "<f8", "float64": "<f8"}


def construct_list_of_attributes(n_dc=3, n_rest=45, n_scale=3, n_rot=4):
    """gaussian_model.py:472-484."""
    names = ["x", "y", "z", "nx", "ny", "nz"]
    names += ["f_dc_%d" % i for i in range(n_dc)]
    names += ["f_rest_%d" % i for i in range(n_rest)]
    names.append("opacity")
    names += ["scale_%d" % i for i in range(n_scale)]
    names += ["rot_%d" % i for i in range(n_rot)]
    return names


def ply_header(n_vertices, names):
    """The header plyfile writes for one `vertex` element of float32 properties on a little-endian host."""
    lines = ["ply", "format binary_little_endian 1.0", "element vertex %d" % n_vertices]
    lines += ["property float %s" % n for n in names]
    lines.append("end_header")
    return ("\n".join(lines) + "\n").encode("ascii")


def _rows(xyz, features_dc, features_rest, opacity, scaling, rotation):
    """[N, 62] fp32 row matrix in file order; features arrive in the model's layout ([N, 1, 3] and [N, 15, 3]) and are
    stored channel-major (`transpose(1, 2).flatten(start_dim=1)`, gaussian_model.py:531-532)."""
    xyz = xyz.detach().float()
    N = xyz.size(0)
    flat = lambda t, w: t.detach().float().reshape(N, w)  # noqa: E731  (explicit widths: N may be 0)
    f_dc = flat(features_dc.detach().transpose(1, 2), features_dc.size(1) * features_dc.size(2))
    f_rest = flat(features_rest.detach().transpose(1, 2), features_rest.size(1) * features_rest.size(2))
    cols = [xyz, torch.zeros_like(xyz), f_dc, f_rest, flat(opacity, 1), flat(scaling, scaling.size(1)),
            flat(rotation, rotation.size(1))]
    return torch.cat(cols, dim=1).contiguous()


def save_ply(path, xyz, features_dc, features_rest, opacity, scaling, rotation):
    """GaussianModel.save_ply: raw (pre-activation) parameters, normals written as zeros."""
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    rows = _rows(xyz, features_dc, features_rest, opacity, scaling, rotation)
    names = construct_list_of_attributes(features_dc.size(1) * features_dc.size(2),
                                         features_rest.size(1) * features_rest.size(2), scaling.size(1), rotation.size(1))
    assert rows.size(1) == len(names)
    host = rows.cpu().numpy().astype("<f4", copy=False)
    with open(path, "wb") as f:
        f.write(ply_header(rows.size(0), names))
        host.tofile(f)


def read_ply_vertices(path):
    """-> (structured numpy array of the `vertex` element, list of property names).  Binary little-endian and ascii
    files with scalar properties are understood (what plyfile writes for these models); list properties are rejected."""
    with open(path, "rb") as f:
        if f.readline().strip() != b"ply":
            raise ValueError("%s: not a PLY file" % path)
        fmt, elements, cur = None, [], None
        while True:
            line = f.readline()
            if not line:
                raise ValueError("%s: truncated PLY header" % path)
            tok = line.decode("ascii").split()
            if not tok or tok[0] == "comment" or tok[0] == "obj_info":
                continue
            if tok[0] == "format":
                fmt = tok[1]
            elif tok[0] == "element":
                cur = {"name": tok[1], "count": int(tok[2]), "props": []}
                elements.append(cur)
            elif tok[0] == "property":
                if tok[1] == "list":
                    raise ValueError("%s: list properties are not supported" % path)
                cur["props"].append((tok[2], _PLY_TYPES[tok[1]]))
            elif tok[0] == "end_header":
                break
        if fmt not in ("binary_little_endian", "ascii"):
            raise ValueError("%s: unsupported PLY format %r" % (path, fmt))
        out = None
        for el in elements:
            dt = np.dtype(el["props"])
            if fmt == "ascii":
                data = np.loadtxt(f, dtype=np.float64, max_rows=el["count"], ndmin=2)
                arr = np.empty(el["count"], dtype=dt)
                for i, (n, _) in enumerate(el["props"]):
                    arr[n] = data[:, i]
            else:
                arr = np.fromfile(f, dtype=dt, count=el["count"])
                if arr.shape[0] != el["count"]:
                    raise ValueError("%s: truncated PLY body" % path)
            if el["name"] == "vertex":
                out = (arr, [n for n, _ in el["props"]])
                break
        if out is None:
            raise ValueError("%s: no vertex element" % path)
        return out


def load_ply_file(path, degree):
    """GaussianModel.load_ply_file (gaussian_model.py:322-355): same return values, shapes and dtypes —
    xyz [N,3] f32, features_dc [N,3,1] f64, features_extra [N,3,(degree+1)^2-1] f64, opacities [N,1] f32,
    scales [N,3] f64, rots [N,4] f64."""
    v, names = read_ply_vertices(path)
    xyz = np.stack((np.asarray(v["x"]), np.asarray(v["y"]), np.asarray(v["z"])), axis=1)
    opacities = np.asarray(v["opacity"])[..., np.newaxis]
    features_dc = np.zeros((xyz.shape[0], 3, 1))
    for c in range(3):
        features_dc[:, c, 0] = np.asarray(v["f_dc_%d" % c])

    def family(prefix):
        fam = sorted((n for n in names if n.startswith(prefix)), key=lambda x: int(x.split("_")[-1]))
        out = np.zeros((xyz.shape[0], len(fam)))
        for i, n in enumerate(fam):
            out[:, i] = np.asarray(v[n])
        return out
    features_extra = family("f_rest_")
    assert features_extra.shape[1] == 3 * (degree + 1) ** 2 - 3
    features_extra = features_extra.reshape((features_extra.shape[0], 3, (degree + 1) ** 2 - 1))
    return xyz, features_dc, features_extra, opacities, family("scale_"), family("rot")


def load_ply(path, degree=3, device="cuda"):
    """GaussianModel.load_ply (:548-558) without the model object: the six raw parameter tensors in the model's layout
    (features [N,1,3] / [N,15,3]), fp32, on `device`.  The column split and the channel-major -> coefficient-major
    transpose run on the device after ONE upload of the row matrix."""
    v, names = read_ply_vertices(path)
    flat = np.empty((v.shape[0], len(names)), dtype=np.float32)
    for i, n in enumerate(names):
        flat[:, i] = v[n]
    rows = torch.from_numpy(flat).to(device)
    col = {n: i for i, n in enumerate(names)}

    def pick(keys):
        return rows[:, [col[k] for k in keys]].contiguous()

    def fam(prefix):
        return sorted((n for n in names if n.startswith(prefix)), key=lambda x: int(x.split("_")[-1]))
    n_coef = (degree + 1) ** 2
    rest = fam("f_rest_")
    assert len(rest) == 3 * n_coef - 3
    N = rows.size(0)
    return (pick(["x", "y", "z"]), pick(["f_dc_0", "f_dc_1", "f_dc_2"]).view(N, 3, 1).transpose(1, 2).contiguous(),
            pick(rest).view(N, 3, n_coef - 1).transpose(1, 2).contiguous(), pick(["opacity"]), pick(fam("scale_")),
            pick(fam("rot")))


def save_point_cloud_bin(path, xyz, features_dc, features_rest, opacity, scaling, rotation):
    """The raw dump at the end of GaussianModel.save_pt (gaussian_model.py:507-517): int32 count, then xyz, the
    concatenated features [N,16,3], opacity, scaling, rotation as fp32 bytes."""
    t = [x.detach().float().cpu().contiguous() for x in (xyz, torch.cat((features_dc, features_rest), dim=1), opacity,
                                                         scaling, rotation)]
    with open(path, "wb") as f:
        f.write(struct.pack("i", t[0].size(0)))
        for x in t:
            f.write(x.numpy().tobytes())


_PT_FILES = ("done_xyz.pt", "done_dc.pt", "done_rest.pt", "done_opacity.pt", "done_scaling.pt", "done_rotation.pt")


def save_pt(path, xyz, features_dc, features_rest, opacity, scaling, rotation):
    """GaussianModel.save_pt (gaussian_model.py:486-517): the six `done_*.pt` tensors (xyz / features / opacity on the
    CPU, scaling and rotation as they are, like the reference) plus `point_cloud.bin`."""
    os.makedirs(path, exist_ok=True)
    torch.save(xyz.detach().cpu(), os.path.join(path, "done_xyz.pt"))
    torch.save(features_dc.detach().cpu(), os.path.join(path, "done_dc.pt"))
    torch.save(features_rest.detach().cpu(), os.path.join(path, "done_rest.pt"))
    torch.save(opacity.detach().cpu(), os.path.join(path, "done_opacity.pt"))
    torch.save(scaling.detach(), os.path.join(path, "done_scaling.pt"))
    torch.save(rotation.detach(), os.path.join(path, "done_rotation.pt"))
    save_point_cloud_bin(os.path.join(path, "point_cloud.bin"), xyz, features_dc, features_rest, opacity, scaling, rotation)


def load_pt(path, device="cpu"):
    """The inner load_pt of save_pt (gaussian_model.py:497-505) / the `done_scaling.pt`, `done_rotation.pt` reads of
    create_from_hier (:398-399): (xyz, features_dc, features_rest, opacity, scaling, rotation)."""
    return tuple(torch.load(os.path.join(path, f), map_location=device).detach() for f in _PT_FILES)


def save_exposures(path, exposure, image_names):
    """scene/__init__.py:165-170: exposure.json = {image_name: 3x4 nested list} of the per-image exposure matrices."""
    data = {name: exposure[i].detach().cpu().numpy().tolist() for i, name in enumerate(image_names)}
    with open(path, "w") as f:
        json.dump(data, f, indent=2)


def load_exposures(path, device="cuda"):
    """create_from_hier's exposure read (gaussian_model.py:376-385): {image_name: fp32 [3,4] tensor} or None."""
    if not os.path.exists(path):
        return None
    with open(path, "r") as f:
        exposures = json.load(f)
    return {name: torch.tensor(exposures[name], dtype=torch.float32, device=device) for name in exposures}


def load_depth_params(path):
    """depth_params.json of graphdeco 3DGS's dataset readers: {image_name: {"scale", "offset"}} as a dict whose entries
    also carry "med_scale", the median of the POSITIVE scales of the file (0 when there are none).  DESIGN.md §3 "Depth
    regularisation"."""
    with open(path, "r") as f:
        params = json.load(f)
    scales = np.array([float(params[k]["scale"]) for k in params], dtype=np.float64)
    med_scale = float(np.median(scales[scales > 0])) if (scales > 0).any() else 0.0
    for k in params:
        params[k]["med_scale"] = med_scale
    return params


def attach_depth_prior(cam, invdepth, depth_params=None, mask=None, device=None):
    """Set `cam.invdepthmap`, `cam.depth_mask` and `cam.depth_reliable` as graphdeco 3DGS's Camera.__init__ does from a
    monocular inverse-depth map ALREADY at render resolution ([H, W] or [1, H, W], H x W = cam.image_height x
    cam.image_width; a tensor or an array; decoding and resizing are the dataset tooling's): negative values are clamped
    to 0 first; with `depth_params` (an entry of load_depth_params) the prior is unreliable when scale < 0.2 med_scale or
    scale > 5 med_scale, which also zeroes the mask, and the map becomes invdepth * scale + offset when scale > 0.
    `mask`: a float map of the same shape, or None for all ones.  The maps are stored as float32 [1, H, W] on `device`
    (default: where `invdepth` is; the trainer wants the parameters' device).  Returns `cam`."""
    H, W = int(cam.image_height), int(cam.image_width)

    def as_map(x, what):
        t = torch.as_tensor(x)
        if t.dim() == 2:
            t = t[None]
        if tuple(t.shape) != (1, H, W):
            raise ValueError("attach_depth_prior: %s has shape %s, the camera renders (1, %d, %d)"
                             % (what, tuple(torch.as_tensor(x).shape), H, W))
        return t.to(device=device if device is not None else t.device, dtype=torch.float32).contiguous()

    inv = as_map(invdepth, "invdepth").clone()
    m = as_map(mask, "mask").clone() if mask is not None else None
    inv[inv < 0] = 0
    reliable = True
    if depth_params is not None:
        scale, offset, med = float(depth_params["scale"]), float(depth_params["offset"]), float(depth_params["med_scale"])
        if scale < 0.2 * med or scale > 5 * med:
            reliable = False
            m = torch.zeros_like(inv) if m is None else m * 0
        if scale > 0:
            inv = inv * scale + offset
    cam.invdepthmap, cam.depth_mask, cam.depth_reliable = inv, m, reliable
    return cam
