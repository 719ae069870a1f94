"""Golden data for the tests that compare against the UNMODIFIED reference itself (oracle/_ref, built by
oracle/build_ref.sh): what each test compared against, stored small enough to keep in tests/golden/.

Arrays a test compares bit for bit are stored as sha256 digests (util.digest); float arrays as a fixed sample of
their elements (util.sample, drawn among the rows of visible Gaussians where most rows are not) or as values at
stored positions among their nonzero elements (util.pick), together with the full tensor's largest magnitude, which
the tests' bars are normalised by.  The inputs are regenerated from their seeds by the tests.

    python tools/make_golden_refext.py cpu OUT_DIR     # learning-rate schedule, deformation cold path
    python tools/make_golden_refext.py gpu OUT_DIR     # reference CUDA extensions and GPU stack (needs a B200)
then copy OUT_DIR/ref_*.npz to tests/golden/."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import ref_ext  # noqa: E402
import util     # noqa: E402

DEV = "cuda:0"


def grab_functions(rel_path, names, ns):
    """exec the named FunctionDefs of a reference source file (oracle/_ref/s3g_ref/<rel_path>) into ns, unmodified"""
    import ast
    path = os.path.join(ref_ext.REF_DIR, "s3g_ref", rel_path)
    for node in ast.walk(ast.parse(open(path).read())):
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns


def picked(out, key, t, k, seed=0):
    """store t's values at up to k positions among its nonzero elements, and the positions"""
    idx = util.pick(t, k, seed)
    out[key + "_idx"] = idx
    out[key + "_s"] = util._np(t).reshape(-1)[idx]


# ---------------------------------------------------------------- CPU
def lr_schedule():
    """test_model_host.test_learning_rates_follow_the_reference_schedule: the reference's update_learning_rate
    (and get_expon_lr_func) driven over the param groups our training_setup builds."""
    import types
    import test_model_host as tm
    ns = {"torch": torch, "nn": torch.nn, "np": np}
    grab_functions(os.path.join("utils", "general_utils.py"), {"get_expon_lr_func"}, ns)
    grab_functions(os.path.join("scene", "gaussian_model.py"), {"update_learning_rate"}, ns)
    m = tm._our_model()
    s, OPT, f = m.spatial_lr_scale, tm.OPT, ns["get_expon_lr_func"]
    ref = types.SimpleNamespace(
        optimizer=types.SimpleNamespace(param_groups=[dict(g) for g in m.optimizer.param_groups]),
        xyz_scheduler_args=f(lr_init=OPT.position_lr_init * s, lr_final=OPT.position_lr_final * s,
                             lr_delay_mult=OPT.position_lr_delay_mult, max_steps=OPT.position_lr_max_steps),
        deformation_scheduler_args=f(lr_init=OPT.deformation_lr_init * s, lr_final=OPT.deformation_lr_final * s,
                                     lr_delay_mult=OPT.deformation_lr_delay_mult, max_steps=OPT.position_lr_max_steps),
        grid_scheduler_args=f(lr_init=OPT.grid_lr_init * s, lr_final=OPT.grid_lr_final * s,
                              lr_delay_mult=OPT.deformation_lr_delay_mult, max_steps=OPT.position_lr_max_steps))
    its, ret, groups = tm.ITERATIONS, [], []
    for it in its:
        ret.append(ns["update_learning_rate"](ref, it))
        groups.append([g["lr"] for g in ref.optimizer.param_groups])
    return dict(iterations=np.array(its), lr=np.array(ret, np.float64), group_lr=np.array(groups, np.float64),
                group_names=np.array([g["name"] for g in ref.optimizer.param_groups]))


def deform_cold():
    """test_deform_cold_host.test_cold_path_equals_reference_module: the reference deform_network's outputs,
    input gradients and parameter gradients for every case."""
    import test_deform_cold_host as tc
    ref_dn, _ = ref_ext.load_ref_deform()
    out = {}
    for cid, flags in zip(tc.IDS, tc.CASES):
        net = tc.make_net(ref_dn, flags)
        base, weights = tc.case_inputs(flags, net)
        a_in = [t.clone().requires_grad_(True) for t in base]
        a = net(*a_in, torch.full((tc.P, 1), 0.4))
        ws = weights(a)
        out[f"{cid}/keys"] = "\n".join(sorted(net.state_dict()))
        out[f"{cid}/outputs"] = np.array([x is not None for x in a])
        sum((x * w).sum() for x, w in zip(a, ws) if x is not None).backward()
        outs = [x for x in a if x is not None]
        grads = [x.grad for x in a_in if x.grad is not None]
        out[f"{cid}/in_grads"] = np.array([x.grad is not None for x in a_in])
        for name, ts in (("out", outs), ("in", grads)):
            out[f"{cid}/{name}_s"] = np.concatenate([util.sample(t, 64) for t in ts])
            out[f"{cid}/{name}_max"] = np.array([float(t.abs().max()) for t in ts])
        params = [(k, p.grad) for k, p in net.named_parameters() if p.grad is not None]
        out[f"{cid}/p_names"] = "\n".join(k for k, _ in params)
        idx = [util.pick(g, 16) for _, g in params]
        out[f"{cid}/p_n"] = np.array([len(i) for i in idx])
        out[f"{cid}/p_idx"] = np.concatenate(idx)
        out[f"{cid}/p_s"] = np.concatenate([g.reshape(-1).numpy()[i] for (_, g), i in zip(params, idx)])
        out[f"{cid}/p_max"] = np.array([float(g.abs().max()) for _, g in params])
    return out


# ---------------------------------------------------------------- GPU
def knn_ext():
    """test_gpu_init.test_distcuda2_matches_oracle_and_reference_extension: the reference distCUDA2."""
    import test_gpu_init as ti
    ref = ref_ext.load_ref_simple_knn()
    return {name: util.digest(ref(pts.to(DEV))) for name, pts in ti.knn_ext_cases()}


def ref_state_record(ref, d, images=False):
    """One forward of the reference extension, kept as its golden record: num_rendered, digests of radii and of the
    internal state check_state_vs compares, and (images=True) a sample and the max of colour and depth."""
    E = torch.Tensor([])
    P, W, H = d["means3D"].shape[0], d["W"], d["H"]
    g = lambda k: d[k].to(DEV).contiguous() if d[k] is not None else E
    R0, rc, rdep, rrad, gb, bb, ib = ref._C.rasterize_gaussians(
        d["bg"].to(DEV), g("means3D"), g("colors_precomp"), g("opacities"), g("scales"), g("rotations"), 1.0,
        g("cov3D_precomp"), d["viewmatrix"].to(DEV), d["projmatrix"].to(DEV), d["tanfovx"], d["tanfovy"], H, W,
        g("shs"), d["sh_degree"], d["campos"].to(DEV), False, False)
    torch.cuda.synchronize()
    rg, rb, ri = ref_ext.decode_geom(gb, P), ref_ext.decode_binning(bb, R0), ref_ext.decode_image(ib, W * H)
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    rec = dict(num_rendered=int(R0), radii=util.digest(rrad), tiles_touched=util.digest(rg["tiles_touched"]),
               point_list=util.digest(rb["point_list"]),
               point_list_tiles=util.digest((rb["point_list_keys"] >> np.uint64(32)).astype(np.uint32)),
               ranges=util.digest(ri["ranges"].reshape(-1, 2)[:tiles]), n_contrib=util.digest(ri["n_contrib"]))
    if images:
        for k, v in (("color", rc), ("depth", rdep)):
            rec[k + "_s"], rec[k + "_max"] = util.sample(v), float(v.abs().max())
    return rec


def raster_bench():
    """test_gpu_raster.test_cuda_matches_reference_extension_at_benchmark_sizes: NRUN runs of the reference
    extension (images; gradients at positions among the visible Gaussians' rows, their mean and run-to-run spread)
    and its internal state."""
    import test_gpu_raster as tr
    ref = ref_ext.load()
    out = {}
    for P, W, H, mode, view in tr.BENCH_CASES:
        cid = tr.bench_case_id(P, W, H, mode, view)
        d, gc, gd = tr.bench_case_inputs(P, W, H, mode, view)
        refs = [util.run_module(ref, d, DEV, gc, gd) for _ in range(tr.NRUN)]
        r = refs[0]
        for k in ("color", "depth"):
            out[f"{cid}/{k}_s"] = util.sample(r[k], tr.IMG_SAMPLE)
            out[f"{cid}/{k}_max"] = float(r[k].abs().max())
        out[f"{cid}/grad_keys"] = " ".join(sorted(r["grads"]))
        vis = r["radii"] > 0
        for k in r["grads"]:
            R = [x["grads"][k].cpu().numpy() for x in refs]
            mean = np.mean(R, axis=0, dtype=np.float64)
            out[f"{cid}/g/{k}_mean_s"] = util.sample(mean, tr.GRAD_SAMPLE, where=util.rows_mask(vis, mean.shape)).astype(np.float32)
            out[f"{cid}/g/{k}_max"] = float(np.abs(R[0]).max())
            out[f"{cid}/g/{k}_spread"] = max(float(np.abs(R[i] - R[j]).max()) for i in range(tr.NRUN) for j in range(i))
        del refs, r
        out.update({f"{cid}/{k}": v for k, v in ref_state_record(ref, d).items()})
    return out


def raster_scale_cams():
    """test_gpu_raster.test_scale_run_cameras_integer_state_matches_reference: the reference extension's
    state and images for the seven other cameras of the scaling run."""
    import test_gpu_raster as tr
    ref = ref_ext.load()
    out = {}
    for rank, d in tr.scale_run_cases():
        rec = ref_state_record(ref, d, images=True)
        out.update({f"rank{rank}/{k}": v for k, v in rec.items()})
    return out


def image_loss():
    """test_gpu_train.test_image_loss_matches_reference_functions_on_gpu: the reference's utils/loss_utils.py
    composed as train.py:395-419, TF32 off in cuDNN."""
    import test_gpu_train as tt
    import make_golden_train as mg
    lu = ref_ext.load_ref_loss_utils()
    torch.backends.cudnn.allow_tf32 = False
    out = {}
    for name, shape, seed in tt.LOSS_CASES:
        img, gt, depth, gt_depth = [t.to(DEV) for t in mg.loss_inputs(*shape, seed)]
        xr = img.clone().requires_grad_(True)
        dr = depth.clone().requires_grad_(True)
        ref = lu.l1_loss(xr, gt) + 0.5 * lu.compute_depth("l2", dr, gt_depth)
        if name == "ssim":
            ref = ref + 0.2 * (1.0 - lu.ssim(xr, gt))
        ref.backward()
        out[name + "/loss"] = float(ref.item())
        for k, t in (("gx", xr.grad), ("gd", dr.grad)):
            out[f"{name}/{k}_s"] = util.sample(t, tt.LOSS_SAMPLE)
            out[f"{name}/{k}_max"] = float(t.abs().max())
    return out


def densify():
    """test_gpu_train.test_densify_prune_reset_match_reference_methods: the reference GaussianModel's densify,
    add_densification_stats, prune, reset_opacity and an Adam step on the test's state."""
    import test_gpu_train as tt
    from s3gaussian_b200.gaussian_model import PARAM_GROUPS, _ATTR
    Ref = ref_ext.load_ref_gaussian_model_class()
    _, ref = tt._pair_of_models(50000, 7, Ref)
    extent, out = 20.0, {}
    torch.manual_seed(123)
    ref.densify(0.0002, 0.005, extent, None, 5, 5, None, None, None)
    out.update({f"densify/{k}": v for k, v in tt.state_record(ref).items()})
    n1 = ref._xyz.shape[0]
    g = torch.Generator(device=DEV).manual_seed(9)
    radii = torch.randint(0, 45, (n1,), device=DEV, generator=g, dtype=torch.int32)
    radii[torch.rand(n1, device=DEV, generator=g) < 0.3] = 0
    vgrad = torch.randn(n1, 3, device=DEV, generator=g) * 1e-3
    vis = radii > 0
    ref.max_radii2D[vis] = torch.max(ref.max_radii2D[vis], radii[vis])
    ref.add_densification_stats(vgrad, vis)
    for a in ("max_radii2D", "denom", "xyz_gradient_accum"):
        out[f"stats/{a}"] = util.digest(getattr(ref, a))
    ref.prune(0.0002, 0.005, extent, 20)
    out.update({f"prune/{k}": v for k, v in tt.state_record(ref).items()})
    ref.reset_opacity()
    out.update({f"reset_opacity/{k}": v for k, v in tt.state_record(ref).items()})
    for n in PARAM_GROUPS:
        pr = getattr(ref, _ATTR[n])
        pr.grad = torch.randn(pr.shape, device=DEV, generator=g) * 0.01
    ref.optimizer.step()
    for n in PARAM_GROUPS:
        p = getattr(ref, _ATTR[n]).detach()
        out[f"adam/{n}_s"], out[f"adam/{n}_max"] = util.sample(p, tt.DENSIFY_SAMPLE), float(p.abs().max())
    return out


def render_stack():
    """test_gpu_deform.test_render_matches_reference_stack_on_gpu: the reference's deform_network, activations,
    eval_sh and CUDA rasterizer (gaussian_renderer/__init__.py:89-166), rgb + feat passes, and the backward."""
    import test_gpu_deform as td
    from s3gaussian_b200 import synthetic as syn
    ref = ref_ext.load()
    ref_deform_network, eval_sh = ref_ext.load_ref_deform()
    out = {}
    for (P, W, H), cid in zip(td.STACK_CASES, td.STACK_IDS):
        cloud, cam, st, gc, gd = td.stack_case(P, W, H)
        theirs = ref_deform_network(ref_ext.ref_deform_args(syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES))
        theirs.deformation_net.set_aabb(*[list(a) for a in syn.WAYMO_AABB])
        theirs.load_state_dict(st, strict=False)
        theirs = util.fill_uncovered(theirs, st).to(DEV)
        xyz = cloud.xyz.to(DEV).requires_grad_(True); sc = cloud.scaling.to(DEV).requires_grad_(True)
        ro = cloud.rotation.to(DEV).requires_grad_(True); op = cloud.opacity.to(DEV).requires_grad_(True)
        shs = cloud.get_features().to(DEV).requires_grad_(True)
        t = torch.full((P, 1), cam.time, device=DEV)
        m3, s2, r2, o2, shf, dx, feat, dshs = theirs(xyz, sc, ro, op, shs, t)
        s_a, r_a, o_a = torch.exp(s2), torch.nn.functional.normalize(r2), torch.sigmoid(o2)
        campos = cam.camera_center.to(DEV)
        dirn = xyz - campos; dirn = dirn / dirn.norm(dim=1, keepdim=True)
        colors = torch.clamp_min(eval_sh(3, shf.transpose(1, 2).view(-1, 3, 16), dirn) + 0.5, 0.0)
        bg = torch.zeros(3, device=DEV)
        rs = util.settings_for(ref, dict(H=H, W=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg,
                                         viewmatrix=cam.world_view_transform, projmatrix=cam.full_proj_transform,
                                         sh_degree=3, campos=cam.camera_center), DEV)
        rast = ref.GaussianRasterizer(rs)
        m2d = torch.zeros_like(xyz, requires_grad=True)
        kw = dict(means3D=m3, means2D=m2d, shs=None, opacities=o_a, scales=s_a, rotations=r_a, cov3D_precomp=None)
        img, radii, dep = rast(colors_precomp=colors, **kw)
        img2, _, _ = rast(colors_precomp=feat, **kw)
        td.stack_loss(img, dep, img2, dx, dshs, gc, gd).backward()
        for k, v in (("render", img), ("depth", dep), ("feat", img2)):
            out[f"{cid}/{k}_s"], out[f"{cid}/{k}_max"] = util.sample(v, td.STACK_IMG), float(v.abs().max())
        out[f"{cid}/radii_s"] = util.sample(radii, 4 * td.STACK_GRAD)
        picked(out, f"{cid}/xyz", xyz.grad, td.STACK_GRAD)
        picked(out, f"{cid}/shs", shs.grad, td.STACK_GRAD)
        names = [k for k, p in theirs.named_parameters() if p.grad is not None]
        out[f"{cid}/param_names"] = " ".join(names)
        for k, p in theirs.named_parameters():
            if p.grad is not None:
                picked(out, f"{cid}/p/{k}", p.grad, td.STACK_PARAM)
    return out


def cold_switch():
    """test_gpu_deform.test_cold_switches_render_through_the_pytorch_path: the reference module's dx and dshs."""
    import test_gpu_deform as td
    ref_dn, _ = ref_ext.load_ref_deform()
    theirs, cloud, cam = td.cold_switch_case(ref_dn)
    theirs = theirs.to(DEV)
    n = cloud.xyz.shape[0]
    xyz, shs = cloud.xyz.to(DEV), cloud.get_features().to(DEV)
    t = torch.full((n, 1), cam.time, device=DEV)
    m3, s2, r2, o2, shf, dx, feat, dshs = theirs(xyz, cloud.scaling.to(DEV), cloud.rotation.to(DEV),
                                                 cloud.opacity.to(DEV), shs, t)
    return {"keys": "\n".join(sorted(theirs.state_dict())), "dx": dx.detach().cpu().numpy(),
            "dshs_s": util.sample(dshs, 1024), "dshs_max": float(dshs.abs().max())}


def main(which, out_dir):
    os.makedirs(out_dir, exist_ok=True)
    jobs = {"cpu": (("ref_lr_schedule", lr_schedule), ("ref_deform_cold", deform_cold)),
            "gpu": (("ref_knn_ext", knn_ext), ("ref_raster_bench", raster_bench),
                    ("ref_raster_scale_cams", raster_scale_cams), ("ref_image_loss", image_loss),
                    ("ref_densify", densify), ("ref_render_stack", render_stack), ("ref_cold_switch", cold_switch))}[which]
    only = sys.argv[3:]
    for name, fn in jobs:
        if only and name not in only:
            continue
        path = os.path.join(out_dir, name + ".npz")
        util.save_golden(path, fn())
        print(path, os.path.getsize(path))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
