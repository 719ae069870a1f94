"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import numpy as np
import torch

from s3gaussian_b200 import synthetic as syn


def scene_inputs(cloud, cam, mode="sh", sh_degree=3, bg=(0.1, 0.2, 0.3), cov_precomp=False):
    """dict of CPU tensors = the arguments of one rasterizer call (post-activation)."""
    d = dict(
        means3D=cloud.xyz.clone(), opacities=cloud.get_opacity().clone(),
        scales=cloud.get_scaling().clone(), rotations=cloud.get_rotation().clone(),
        shs=cloud.get_features().clone() if mode == "sh" else None,
        colors_precomp=torch.sigmoid(cloud.features_dc[:, 0]).clone() if mode != "sh" else None,
        viewmatrix=cam.world_view_transform.clone(), projmatrix=cam.full_proj_transform.clone(),
        campos=cam.camera_center.clone(), bg=torch.tensor(bg, dtype=torch.float32),
        W=cam.image_width, H=cam.image_height, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
        sh_degree=sh_degree, cov3D_precomp=None)
    if cov_precomp:
        d["cov3D_precomp"] = cov3d_from(d["scales"], d["rotations"])
        d["scales"] = None
        d["rotations"] = None
    return d


def cov3d_from(scales, rot):
    """upper-triangular Sigma = R S^2 R^T, [P,6] (host torch, float64 -> float32)."""
    r, x, y, z = [rot[:, i].double() for i in range(4)]
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], 1).view(-1, 3, 3)
    L = R * scales.double()[:, None, :]
    S = L @ L.transpose(1, 2)
    return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1).float()


def settings_for(mod, d, dev, debug=False):
    return mod.GaussianRasterizationSettings(
        image_height=d["H"], image_width=d["W"], tanfovx=d["tanfovx"], tanfovy=d["tanfovy"],
        bg=d["bg"].to(dev), scale_modifier=1.0, viewmatrix=d["viewmatrix"].to(dev),
        projmatrix=d["projmatrix"].to(dev), sh_degree=d["sh_degree"], campos=d["campos"].to(dev),
        prefiltered=False, debug=debug)


TENSOR_KEYS = ("means3D", "opacities", "scales", "rotations", "shs", "colors_precomp", "cov3D_precomp")


def run_module(mod, d, dev, grad_color=None, grad_depth=None):
    """One forward (+ backward when grads are given) through a diff_gaussian_rasterization-like
    module.  Returns dict(color, radii, depth, grads{...}, ctx-free)."""
    t = {k: (d[k].to(dev).clone().requires_grad_(grad_color is not None) if d[k] is not None else None)
         for k in TENSOR_KEYS}
    m2d = torch.zeros_like(t["means3D"], requires_grad=grad_color is not None)
    rast = mod.GaussianRasterizer(settings_for(mod, d, dev))
    color, radii, depth = rast(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"],
                               shs=t["shs"], colors_precomp=t["colors_precomp"], scales=t["scales"],
                               rotations=t["rotations"], cov3D_precomp=t["cov3D_precomp"])
    out = dict(color=color.detach(), radii=radii.detach(), depth=depth.detach(), grads={})
    if grad_color is not None:
        loss = (color * grad_color.to(dev)).sum() + (depth * grad_depth.to(dev)).sum()
        loss.backward()
        out["grads"] = {k: t[k].grad.detach() for k in TENSOR_KEYS if t[k] is not None and t[k].grad is not None}
        out["grads"]["means2D"] = m2d.grad.detach()
    return out


def ours_forward_state(d, dev):
    """Forward through our autograd Function keeping the opaque buffers; returns
    (color, radii, depth, R, views) where views is a dict of numpy arrays of our state."""
    from s3gaussian_b200 import _lib
    from s3gaussian_b200 import diff_gaussian_rasterization as ours

    class Ctx:
        def save_for_backward(self, *a):
            self.saved = a

        def mark_non_differentiable(self, *a):
            pass

    E = torch.Tensor([])
    g = lambda k: d[k].to(dev).contiguous() if d[k] is not None else E
    ctx = Ctx()
    color, radii, depth = ours._RasterizeGaussians.forward(
        ctx, g("means3D"), torch.zeros_like(g("means3D")), g("shs"), g("colors_precomp"), g("opacities"),
        g("scales"), g("rotations"), g("cov3D_precomp"), settings_for(ours, d, dev))
    torch.cuda.synchronize()
    R = ctx.num_rendered
    P, W, H = d["means3D"].shape[0], d["W"], d["H"]
    bufs = {0: ctx.saved[7], 1: ctx.saved[8], 2: ctx.saved[9]}

    def view(bid, name, dt):
        off, eb, cnt = _lib.state_field(bid, name, P, R, W, H)
        buf = bufs[bid]
        if buf.numel() == 0 or cnt == 0:
            return np.zeros(0, dt)
        base = buf.data_ptr()
        a = ((base + 127) & ~127) - base + off
        return buf.cpu().numpy()[a:a + eb * cnt].view(dt).copy()

    views = dict(
        xyAB=view(0, "xyAB", np.float32).reshape(-1, 4), Cod=view(0, "Cod", np.float32).reshape(-1, 4),
        rgb=view(0, "rgb", np.float32).reshape(-1, 4), tiles_touched=view(0, "tiles_touched", np.uint32),
        point_list=view(1, "point_list", np.uint32) if R > 0 else np.zeros(0, np.uint32),
        ranges=view(2, "ranges", np.uint32).reshape(-1, 2), n_contrib=view(2, "n_contrib", np.uint32),
        final_T=view(2, "final_T", np.float32))
    # The sorted tile ids (high 32 bits of the reference's sorted keys) are not materialised any more: the per-tile
    # ranges come from the tile histogram.  Rebuild them from the ranges: tile t owns [start, end) of the list; the
    # tests compare this against the reference's keys, which also checks that the ranges tile the list exactly.
    rng = views["ranges"].astype(np.int64)
    lens = rng[:, 1] - rng[:, 0]
    tiles = np.full(R, 0xFFFFFFFF, np.uint32)
    nz = np.nonzero(lens > 0)[0]
    if nz.size and int(lens.sum()) == R and np.array_equal(rng[nz, 0], np.cumsum(lens[nz]) - lens[nz]):
        tiles = np.repeat(nz.astype(np.uint32), lens[nz])
    views["point_list_tiles"] = tiles
    return color, radii, depth, R, views


def oracle_run(oracle_mod, d, grad_color=None, grad_depth=None):
    o = oracle_mod.Oracle()
    n = lambda k: None if d[k] is None else d[k].numpy()
    color, radii, depth = o.forward(
        bg=d["bg"].numpy(), W=d["W"], H=d["H"], means3D=n("means3D"), opacities=n("opacities"),
        viewmatrix=d["viewmatrix"].numpy(), projmatrix=d["projmatrix"].numpy(), campos=d["campos"].numpy(),
        tanfovx=d["tanfovx"], tanfovy=d["tanfovy"], sh_degree=d["sh_degree"], shs=n("shs"),
        colors_precomp=n("colors_precomp"), scales=n("scales"), rotations=n("rotations"),
        cov3D_precomp=n("cov3D_precomp"))
    out = dict(color=color, radii=radii, depth=depth, R=o.R, geometry=o.geometry(), binning=o.binning(),
               image=o.image_state(), grads=None)
    if grad_color is not None:
        out["grads"] = o.backward(grad_color.numpy(), grad_depth.numpy())
    return out


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def elementwise(a, b, rtol=1e-4, atol=0.0):
    """Element-wise closeness |a-b| <= rtol*|b| + atol (north_star's "1e-4 relative fp32" read literally, plus an
    absolute floor the caller states and justifies).  Returns (fraction of elements outside, worst excess ratio
    |a-b| / (rtol*|b| + atol), index of the worst element)."""
    a = np.asarray(a, np.float64).reshape(-1)
    b = np.asarray(b, np.float64).reshape(-1)
    lim = rtol * np.abs(b) + atol
    err = np.abs(a - b)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(lim > 0, err / lim, np.where(err > 0, np.inf, 0.0))
    i = int(np.argmax(ratio)) if ratio.size else 0
    return float((ratio > 1.0).mean()) if ratio.size else 0.0, float(ratio[i]) if ratio.size else 0.0, i


def grad_atol(ref_run_a, ref_run_b, floor_of_max=1e-6):
    """Absolute floor for element-wise gradient checks: the reference's OWN run-to-run spread on this input
    (its backward accumulates with unordered fp32 atomics, backward.cu:550-587) times 4, but at least
    `floor_of_max` of the tensor's largest magnitude (fp32 accumulation noise of a sum of hundreds of terms)."""
    a = np.asarray(ref_run_a, np.float64)
    b = np.asarray(ref_run_b, np.float64)
    return max(4.0 * float(np.abs(a - b).max()), floor_of_max * float(np.abs(a).max()))


def _np(a):
    return a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)


def digest(a):
    """sha256 of an array's bytes: stored in place of a large array that a test compares bit for bit."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(_np(a)).tobytes()).hexdigest()


def sample(a, k=256, seed=0, where=None):
    """k elements of the flattened array at positions fixed by (size, k, seed): stored in place of a large float array
    so that a test compares the same positions of its own result.  `where` (a mask of a's shape, e.g. the rows of
    visible Gaussians, which both sides must agree on) restricts the draw to the positions it marks."""
    a = _np(a).reshape(-1)
    pos = np.arange(a.size) if where is None else np.flatnonzero(_np(where).reshape(-1))
    if pos.size <= k:
        return a[pos].copy()
    return a[pos[np.sort(np.random.default_rng(seed).choice(pos.size, k, replace=False))]]


def rows_mask(rows, shape):
    """bool mask of `shape` marking every element of the rows (first axis) where `rows` is true"""
    rows = _np(rows).astype(bool)
    return np.broadcast_to(rows.reshape((-1,) + (1,) * (len(shape) - 1)), shape)


def save_golden(path, record):
    """Write a dict of arrays, numbers and strings as one .npz: an index (JSON) and one flat array per dtype.  A
    record of hundreds of small entries would otherwise spend more on per-entry headers than on its values."""
    import json
    index, flat = {}, {}
    for k, v in record.items():
        if isinstance(v, str):
            index[k] = v
            continue
        a = np.asarray(v)
        key = a.dtype.str
        off = sum(x.size for x in flat.setdefault(key, []))
        flat[key].append(a.reshape(-1))
        index[k] = [key, off, list(a.shape)]
    np.savez_compressed(path, index=np.frombuffer(json.dumps(index).encode(), np.uint8),
                        **{"d" + k.replace("<", "l").replace(">", "b").replace("|", "n"): np.concatenate(v)
                           for k, v in flat.items()})


def load_golden(path):
    """dict of what save_golden() stored: strings as str, everything else as numpy arrays of the stored shape"""
    import json
    z = np.load(path)
    index = json.loads(z["index"].tobytes().decode())
    flat = {k: z[k] for k in z.files if k != "index"}
    out = {}
    for k, v in index.items():
        if isinstance(v, str):
            out[k] = v
        else:
            key, off, shape = v
            n = int(np.prod(shape)) if shape else 1
            out[k] = flat["d" + key.replace("<", "l").replace(">", "b").replace("|", "n")][off:off + n].reshape(shape)
    return out


def fill_uncovered(net, state, seed=6):
    """Draw the parameters of `net` that the seeded `state` does not cover (time net, static_mlp) from a generator of
    their own, in name order, so that the reference's network and ours get the same weights."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for k, p in sorted(net.named_parameters()):
            if k not in state:
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return net


def pick(a, k, seed=0):
    """int32 positions of up to k nonzero elements of the flattened array: stored with the values there when the two
    sides may disagree on which elements are zero"""
    nz = np.flatnonzero(_np(a).reshape(-1))
    if nz.size > k:
        nz = nz[np.sort(np.random.default_rng(seed).choice(nz.size, k, replace=False))]
    return nz.astype(np.int32)


def relerr_sampled(ours, ref_sample, ref_absmax, k=256, seed=0, where=None):
    """relerr() restricted to the stored sample positions, normalised by the full reference tensor's max."""
    s = sample(ours, k, seed, where).astype(np.float64)
    return float(np.abs(s - ref_sample).max() / (float(ref_absmax) + 1e-30)) if s.size else 0.0


def seeded_grads(d, seed=1):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(3, d["H"], d["W"], generator=g), torch.randn(1, d["H"], d["W"], generator=g))


# ---- the reference's fine-stage render() code path, assembled from ITS OWN modules ----------
class RefFineStack:
    """gaussian_renderer/__init__.py:89-166 with the reference's deform_network (PyTorch), activations,
    eval_sh and CUDA rasterizer, all from oracle/_ref.  Used as the checker and as bench.py's reference arm
    for the fine-stage workload."""

    def __init__(self, cloud, state, dev, resolution, multires):
        import ref_ext
        from s3gaussian_b200 import synthetic as syn
        self.ref = ref_ext.load()
        deform_network, self.eval_sh = ref_ext.load_ref_deform()
        net = deform_network(ref_ext.ref_deform_args(resolution, multires))
        net.deformation_net.set_aabb(*[list(a) for a in syn.WAYMO_AABB])
        net.load_state_dict(state, strict=False)
        self.net = net.to(dev)
        self.dev = dev
        T = lambda t: t.to(dev).clone().requires_grad_(True)
        self.xyz, self.scaling, self.rotation, self.opacity = T(cloud.xyz), T(cloud.scaling), T(cloud.rotation), T(cloud.opacity)
        self.f_dc, self.f_rest = T(cloud.features_dc), T(cloud.features_rest)
        self.P = cloud.xyz.shape[0]

    def leaves(self):
        return [self.xyz, self.scaling, self.rotation, self.opacity, self.f_dc, self.f_rest] + list(self.net.parameters())

    def render(self, cam, bg, render_feat=True):
        dev, P = self.dev, self.P
        shs = torch.cat((self.f_dc, self.f_rest), dim=1)
        t = torch.full((P, 1), float(cam.time), device=dev)
        m3, sc, ro, op, shf, dx, feat, dshs = self.net(self.xyz, self.scaling, self.rotation, self.opacity, shs, t)
        s_a, r_a, o_a = torch.exp(sc), torch.nn.functional.normalize(ro), torch.sigmoid(op)
        campos = cam.camera_center.to(dev)
        dirn = self.xyz - campos.repeat(P, 1)
        dirn = dirn / dirn.norm(dim=1, keepdim=True)
        colors = torch.clamp_min(self.eval_sh(3, shf.transpose(1, 2).view(-1, 3, 16), dirn) + 0.5, 0.0)
        rs = self.ref.GaussianRasterizationSettings(
            image_height=cam.image_height, image_width=cam.image_width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg,
            scale_modifier=1.0, viewmatrix=cam.world_view_transform.to(dev), projmatrix=cam.full_proj_transform.to(dev),
            sh_degree=3, campos=campos, prefiltered=False, debug=False)
        rast = self.ref.GaussianRasterizer(rs)
        m2d = torch.zeros_like(self.xyz, requires_grad=True)
        img, radii, dep = rast(means3D=m3, means2D=m2d, shs=None, colors_precomp=colors, opacities=o_a, scales=s_a,
                               rotations=r_a, cov3D_precomp=None)
        out = {"render": img, "radii": radii, "depth": dep, "dx": dx, "dshs": dshs, "viewspace_points": m2d}
        if render_feat:
            img2, _, _ = rast(means3D=m3, means2D=m2d, shs=None, colors_precomp=feat, opacities=o_a, scales=s_a,
                              rotations=r_a, cov3D_precomp=None)
            out["feat"] = img2
        return out
