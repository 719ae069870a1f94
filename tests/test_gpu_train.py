"""GPU parity of the training-step kernels (run with -m gpu): fused image loss, multi-tensor Adam,
densification statistics - through the C ABI, against (1) tests/golden/train_*.npz = outputs of the
REAL reference code, (2) the oracle at sizes the goldens do not cover, (3) torch.optim.Adam itself."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_golden_train as mg                                    # noqa: E402 (input generators only)
from test_oracle_train import GOLD, LOSS_GOLD, load_loss_case, rel  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("path", LOSS_GOLD, ids=[os.path.basename(p)[11:-4] for p in LOSS_GOLD])
def test_image_loss_matches_reference_golden(path, built_lib):
    from s3gaussian_b200 import losses
    z, img, gt, depth, gt_depth = load_loss_case(path)
    img = img.to(DEV).requires_grad_(True)
    depth = depth.to(DEV).requires_grad_(True)
    l1, ss, dl2 = losses.image_loss_terms(img, gt.to(DEV), depth, gt_depth.to(DEV))
    loss = l1 + 0.5 * dl2 + 0.2 * (1.0 - ss)
    loss.backward()
    assert abs(l1.item() - float(z["l1"])) < 1e-6
    assert abs(ss.item() - float(z["ssim"])) < 1e-5
    assert abs(dl2.item() - float(z["depth_l2"])) < 1e-6
    assert abs(loss.item() - float(z["loss"])) < 1e-5
    assert rel(img.grad.cpu(), z["g_image"]) < 1e-4
    assert rel(depth.grad.cpu(), z["g_depth"]) < 1e-5
    # the reference-named wrappers give the same numbers one at a time
    assert abs(losses.l1_loss(img.detach(), gt.to(DEV)).item() - float(z["l1"])) < 1e-6
    assert abs(losses.ssim(img.detach(), gt.to(DEV)).item() - float(z["ssim"])) < 1e-5
    assert abs(losses.compute_depth("l2", depth.detach(), gt_depth.to(DEV)).item() - float(z["depth_l2"])) < 1e-6


def test_image_loss_full_size_against_oracle_and_properties(built_lib):
    from oracle import train_oracle as tro
    from s3gaussian_b200 import losses
    img, gt, depth, gt_depth = mg.loss_inputs(1, 3, 1280, 1920, 5)
    img, gt, depth, gt_depth = [t.to(DEV) for t in (img, gt, depth, gt_depth)]
    x = img.clone().requires_grad_(True)
    d = depth.clone().requires_grad_(True)
    ours = losses.training_loss(x, gt, d, gt_depth)
    ours.backward()
    xo = img.double().requires_grad_(True)
    do = depth.double().requires_grad_(True)
    ref = tro.training_loss(xo, gt.double(), do, gt_depth.double())
    ref.backward()
    assert abs(ours.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item()))
    assert rel(x.grad, xo.grad) < 1e-4
    assert rel(d.grad, do.grad) < 1e-5
    # ssim(x, x) == 1, zero gradient; l1 symmetric
    y = gt.clone().requires_grad_(True)
    l1, ss, _ = losses.image_loss_terms(y, gt)
    assert abs(ss.item() - 1.0) < 1e-6 and l1.item() == 0.0
    ss.backward()
    assert float(y.grad.abs().max()) < 1e-9
    assert losses.l1_loss(img, gt).item() == losses.l1_loss(gt, img).item()


def _groups(ps):
    groups = {}
    for (name, _, lr), p in zip(mg.ADAM_SHAPES, ps):
        groups.setdefault(name, {"params": [], "lr": lr, "name": name})["params"].append(p)
    return list(groups.values())


def test_fused_adam_matches_reference_golden(built_lib):
    from s3gaussian_b200.optim import FusedAdam
    z = np.load(os.path.join(GOLD, "train_adam.npz"))
    params, grads = mg.adam_inputs(int(z["seed"]), int(z["steps"]))
    ps = [torch.nn.Parameter(p.clone().to(DEV)) for p in params]
    opt = FusedAdam(_groups(ps), lr=0.0, eps=1e-15)
    for s, gs in enumerate(grads):
        for (name, _, _), p, g in zip(mg.ADAM_SHAPES, ps, gs):
            p.grad = None if name == "nograd" else g.clone().to(DEV)
        if s == 2:
            for gr in opt.param_groups:
                if gr["name"] == "xyz":
                    gr["lr"] = 1.0e-4
        opt.step()
        for i, p in enumerate(ps):
            assert rel(p.detach().cpu(), z[f"p{i}_s{s}"]) < 2e-6, (mg.ADAM_SHAPES[i][0], s)
    for i, p in enumerate(ps):
        st = opt.state.get(p, {})
        if mg.ADAM_SHAPES[i][0] == "nograd":
            assert not st
            continue
        assert rel(st["exp_avg"].cpu(), z[f"m{i}"]) < 2e-6 and rel(st["exp_avg_sq"].cpu(), z[f"v{i}"]) < 2e-6
        assert float(st["step"]) == 3.0


def test_fused_adam_matches_torch_adam_many_tensors_and_state_surgery(built_lib):
    """> 40 tensors (several launches), an unaligned parameter, sizes around the 4096-element chunk, and
    the reference's optimizer-state surgery (prune + cat, scene/gaussian_model.py:411-470) on the state dict."""
    from s3gaussian_b200.optim import FusedAdam
    g = torch.Generator(device=DEV).manual_seed(3)
    sizes = [1, 3, 4095, 4096, 4097, 8192, 12289, 100003] + [257 + 13 * i for i in range(40)] + [(200000, 3), (200000, 15, 3)]
    base = []
    for s in sizes:
        shape = s if isinstance(s, tuple) else (s,)
        base.append(torch.randn(*shape, device=DEV, generator=g))
    storage = torch.randn(5001, device=DEV, generator=g)
    base.append(storage[1:])                                   # 4-byte offset: not 16-byte aligned
    ours = [torch.nn.Parameter(b.clone() if b.data_ptr() % 16 == 0 else b) for b in base]
    ours[-1] = torch.nn.Parameter(storage.clone()[1:])
    theirs = [torch.nn.Parameter(b.clone()) for b in base]
    oa = FusedAdam([{"params": [p], "lr": 1e-3 * (1 + i % 3), "name": str(i)} for i, p in enumerate(ours)], lr=0.0, eps=1e-15)
    ta = torch.optim.Adam([{"params": [p], "lr": 1e-3 * (1 + i % 3), "name": str(i)} for i, p in enumerate(theirs)], lr=0.0, eps=1e-15)
    for step in range(4):
        for po, pt in zip(ours, theirs):
            gr = torch.randn(po.shape, device=DEV, generator=g) * 0.01
            po.grad, pt.grad = gr.clone(), gr.clone()
        oa.step(); ta.step()
    for i, (po, pt) in enumerate(zip(ours, theirs)):
        assert rel(po, pt) < 2e-6, i
        assert rel(oa.state[po]["exp_avg"], ta.state[pt]["exp_avg"]) < 2e-6
        assert rel(oa.state[po]["exp_avg_sq"], ta.state[pt]["exp_avg_sq"]) < 2e-6
    # prune every other row of the [200000,3] tensor and append 100 rows, on both optimizers, then step again
    def surgery(opt, plist, idx):
        group = opt.param_groups[idx]
        p = group["params"][0]
        st = opt.state.get(p)
        mask = torch.arange(p.shape[0], device=DEV) % 2 == 0
        ext = torch.ones(100, 3, device=DEV)
        st["exp_avg"] = torch.cat((st["exp_avg"][mask], torch.zeros_like(ext)))
        st["exp_avg_sq"] = torch.cat((st["exp_avg_sq"][mask], torch.zeros_like(ext)))
        del opt.state[p]
        newp = torch.nn.Parameter(torch.cat((p[mask], ext)).requires_grad_(True))
        group["params"][0] = newp
        opt.state[newp] = st
        plist[idx] = newp
    k = len(sizes) - 2
    surgery(oa, ours, k); surgery(ta, theirs, k)
    gr = torch.randn(ours[k].shape, device=DEV, generator=g)
    for plist in (ours, theirs):
        for p in plist:
            p.grad = None
    ours[k].grad, theirs[k].grad = gr.clone(), gr.clone()
    oa.step(); ta.step()
    assert rel(ours[k], theirs[k]) < 2e-6
    sd = oa.state_dict()
    assert set(sd["state"][k].keys()) == {"step", "exp_avg", "exp_avg_sq"}


def test_densify_stats_matches_reference_golden(built_lib):
    from s3gaussian_b200.optim import add_densification_stats
    z = np.load(os.path.join(GOLD, "train_densify_stats.npz"))
    radii, vgrad, accum, denom, max_radii = [t.to(DEV) for t in mg.stats_inputs(int(z["P"]), int(z["seed"]))]
    add_densification_stats(vgrad, radii, accum, denom, max_radii)
    assert rel(accum.cpu(), z["accum"]) < 1e-6
    assert np.array_equal(denom.cpu().numpy(), z["denom"])
    assert np.array_equal(max_radii.cpu().numpy(), z["max_radii2D"])


LOSS_CASES = [("ssim", (2, 3, 640, 960), 9), ("l1_depth", (2, 3, 640, 960), 10), ("l1_depth_odd", (1, 3, 37, 53), 10)]
LOSS_SAMPLE = 1024


def test_image_loss_matches_reference_functions_on_gpu(built_lib):
    """The reference's own l1_loss / ssim / compute_depth (cuDNN depthwise convs, TF32 off) on the same GPU, composed
    as train.py:395-419: tests/golden/ref_image_loss.npz holds its loss and, at fixed positions, its gradients
    (tools/make_golden_refext.py)."""
    from s3gaussian_b200 import losses
    import util
    z = util.load_golden(os.path.join(GOLD, "ref_image_loss.npz"))
    for name, shape, seed in LOSS_CASES:
        img, gt, depth, gt_depth = [t.to(DEV) for t in mg.loss_inputs(*shape, seed)]
        x = img.clone().requires_grad_(True)
        d = depth.clone().requires_grad_(True)
        if name == "ssim":
            ours = losses.training_loss(x, gt, d, gt_depth)
            bars = (1e-5, 1e-4, 1e-5)
        else:
            # lambda_dssim == 0 (train.py:418 does not evaluate SSIM then): the stencil-free kernels, odd sizes included
            ours = losses.training_loss(x, gt, d, gt_depth, lambda_dssim=0.0, lambda_depth=0.5)
            bars = (1e-6, 1e-6, 1e-5)
        ours.backward()
        assert abs(ours.item() - float(z[name + "/loss"])) < bars[0], name
        assert util.relerr_sampled(x.grad, z[name + "/gx_s"], z[name + "/gx_max"], LOSS_SAMPLE) < bars[1], name
        assert util.relerr_sampled(d.grad, z[name + "/gd_s"], z[name + "/gd_max"], LOSS_SAMPLE) < bars[2], name
        if name != "ssim":
            l1, ss, dl2 = losses.image_loss_terms(x, gt, d, gt_depth, with_ssim=False)
            assert float(ss) == 0.0


def test_plane_regulation_matches_reference_golden(built_lib):
    from s3gaussian_b200 import regulation
    z = np.load(os.path.join(GOLD, "train_plane_reg.npz"))
    levels = [[p.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True) for p in lv]
              for lv in mg.reg_inputs(int(z["seed"]))]
    total = regulation.compute_regulation(levels, 0.01, 0.0001, 0.0001)
    (3.0 * total).backward()
    assert abs(total.item() - float(z["total"])) < 2e-6 * abs(float(z["total"]))
    for l, lv in enumerate(levels):
        for k, p in enumerate(lv):
            assert rel(p.grad.cpu(), 3.0 * z[f"g{l}_{k}"]) < 1e-5, (l, k)
    one = levels[0][2]
    from oracle import train_oracle as tro
    assert abs(regulation.compute_plane_smoothness(one).item() - tro.plane_smoothness(one.detach().cpu().double()).item()) < 1e-6


def test_plane_regulation_full_size_and_adam_on_channels_last_planes(built_lib):
    """The shipped HexPlane (4 levels, 142.9 MB): regulariser vs the oracle on the GPU, then one FusedAdam step
    on the channels_last planes vs torch.optim.Adam."""
    from oracle import train_oracle as tro
    from s3gaussian_b200 import regulation, synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    from s3gaussian_b200.optim import FusedAdam
    import ref_ext
    net = deform_network(ref_ext.ref_deform_args(syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES)).to(DEV)
    grids = net.deformation_net.grid.grids
    g = torch.Generator(device=DEV).manual_seed(1)
    with torch.no_grad():
        for lv in grids:
            for p in lv:
                p.add_(0.05 * torch.randn(p.shape, device=DEV, generator=g).contiguous(memory_format=torch.channels_last))
    total = regulation.compute_regulation(grids, 0.01, 0.0001, 0.0001)
    total.backward()
    ref_planes = [[p.detach().double().requires_grad_(True) for p in lv] for lv in grids]
    ref = tro.compute_regulation(ref_planes, 0.01, 0.0001, 0.0001)
    ref.backward()
    assert abs(total.item() - ref.item()) < 1e-5 * abs(ref.item())
    for lv, rlv in zip(grids, ref_planes):
        for p, r in zip(lv, rlv):
            assert p.grad.stride() == p.stride()
            assert rel(p.grad, r.grad) < 1e-5
    planes = [p for lv in grids for p in lv]
    clones = [torch.nn.Parameter(p.detach().clone()) for p in planes]
    for c, p in zip(clones, planes):
        c.grad = p.grad.clone()
    FusedAdam([{"params": planes, "lr": 1.6e-3, "name": "grid"}], lr=0.0, eps=1e-15).step()
    torch.optim.Adam([{"params": clones, "lr": 1.6e-3, "name": "grid"}], lr=0.0, eps=1e-15).step()
    for c, p in zip(clones, planes):
        assert rel(p, c) < 2e-6


# ---- densify / prune against the reference's own methods ---------------------------------------
class _Params:
    """Stand-in for the reference model in _pair_of_models when only the optimizer set-up is needed."""


def _pair_of_models(P, seed, twin_cls=_Params):
    """Our GaussianModel and a twin of class twin_cls (tools/make_golden_refext.py passes the reference's
    GaussianModel method bodies) over identical tensors, optimizer state and densification statistics."""
    from s3gaussian_b200.gaussian_model import GaussianModel, default_optimization_params, PARAM_GROUPS, _ATTR
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    xyz = r(P, 3) * 10
    scaling = torch.log(torch.exp(r(P, 3) * 0.9 - 2.0))          # scales straddle percent_dense * extent
    ours = GaussianModel(3).create_from_tensors(xyz, r(P, 1, 3), r(P, 15, 3) * 0.1, scaling, r(P, 4), r(P, 1) * 2)
    opt_args = default_optimization_params()
    ours.training_setup(opt_args)
    ref = twin_cls()
    for name in PARAM_GROUPS:
        setattr(ref, _ATTR[name], torch.nn.Parameter(getattr(ours, _ATTR[name]).detach().clone().requires_grad_(True)))
    ref.percent_dense = opt_args.percent_dense
    ref._deformation_table = torch.ones(P, dtype=torch.bool, device=DEV)
    ref.optimizer = torch.optim.Adam([{"params": [getattr(ref, _ATTR[n])], "lr": gr["lr"], "name": n}
                                      for n, gr in ((n, ours._group(n)) for n in PARAM_GROUPS)], lr=0.0, eps=1e-15)
    # two optimizer steps on the twin, then copy its state into ours bit for bit
    for _ in range(2):
        for n in PARAM_GROUPS:
            p = getattr(ref, _ATTR[n])
            p.grad = torch.randn(p.shape, device=DEV, generator=g) * 0.01
        ref.optimizer.step()
    for n in PARAM_GROUPS:
        po, pr = getattr(ours, _ATTR[n]), getattr(ref, _ATTR[n])
        po.data.copy_(pr.data)
        st = ref.optimizer.state[pr]
        ours.optimizer.state[po] = {"step": st["step"].clone(), "exp_avg": st["exp_avg"].clone(),
                                    "exp_avg_sq": st["exp_avg_sq"].clone()}
        pr.grad = None
    acc = torch.rand(P, 1, device=DEV, generator=g) * 6e-4
    den = torch.randint(0, 4, (P, 1), device=DEV, generator=g).float()        # zeros -> nan -> 0 path
    mr = torch.randint(0, 40, (P,), device=DEV, generator=g).float()
    for m in (ours, ref):
        m.xyz_gradient_accum, m.denom, m.max_radii2D = acc.clone(), den.clone(), mr.clone()
        m._deformation_accum = torch.zeros(P, 3, device=DEV)
    return ours, ref


def state_record(m):
    """digest of every parameter, its Adam moments and step, and the densification statistics of model m (ours or
    the reference's): what the densify / prune / reset steps are compared by"""
    import util
    from s3gaussian_b200.gaussian_model import PARAM_GROUPS, _ATTR
    rec = {}
    for n in PARAM_GROUPS:
        p = getattr(m, _ATTR[n])
        st = m.optimizer.state.get(p)
        rec[n] = util.digest(p.data) + str(tuple(p.shape))
        rec[n + ".adam"] = "none" if st is None else \
            util.digest(st["exp_avg"]) + util.digest(st["exp_avg_sq"]) + str(float(st["step"]))
    for a in ("xyz_gradient_accum", "denom", "max_radii2D", "_deformation_accum", "_deformation_table"):
        rec[a] = util.digest(getattr(m, a))
    return rec


def _assert_same_state(ours, z, what):
    from s3gaussian_b200.gaussian_model import PARAM_GROUPS, _ATTR
    for k, v in state_record(ours).items():
        assert v == str(z[f"{what}/{k}"]), (what, k)
    for n in PARAM_GROUPS:
        assert ours._group(n)["params"][0] is getattr(ours, _ATTR[n])


DENSIFY_SAMPLE = 512


def test_densify_prune_reset_match_reference_methods(built_lib):
    """Our densify / stats / prune / reset_opacity / Adam step against the reference's own GaussianModel methods run on
    the same state: tests/golden/ref_densify.npz holds the reference's state after each step (digests, bit for bit)
    and its parameters after the last Adam step (sampled) (tools/make_golden_refext.py)."""
    import util
    from s3gaussian_b200.gaussian_model import PARAM_GROUPS, _ATTR
    z = util.load_golden(os.path.join(GOLD, "ref_densify.npz"))
    P = 50000
    ours, _ = _pair_of_models(P, 7)
    extent = 20.0
    # densify (clone + split), the generator state the reference saw for the torch.normal inside densify_and_split
    torch.manual_seed(123)
    ours.densify(0.0002, 0.005, extent, None)
    assert ours._xyz.shape[0] > P                      # the case is not degenerate
    _assert_same_state(ours, z, "densify")
    n1 = ours._xyz.shape[0]
    # statistics for the next round (ours: fused kernel; reference: its own method + train.py:490)
    g = torch.Generator(device=DEV).manual_seed(9)
    radii = torch.randint(0, 45, (n1,), device=DEV, generator=g, dtype=torch.int32)
    radii[torch.rand(n1, device=DEV, generator=g) < 0.3] = 0
    vgrad = torch.randn(n1, 3, device=DEV, generator=g) * 1e-3
    acc = ours.xyz_gradient_accum.clone()
    ours.densification_step(vgrad, radii)
    assert util.digest(ours.max_radii2D) == str(z["stats/max_radii2D"]) and util.digest(ours.denom) == str(z["stats/denom"])
    # the reference's accumulation (add_densification_stats, one torch statement) on the same device: bit for bit
    # what it stored; ours within 1e-6 (the fused kernel's norm differs in the last ulp), then re-synced for bit tests
    vis = radii > 0
    acc[vis] += torch.norm(vgrad[vis, :2], dim=-1, keepdim=True)
    assert util.digest(acc) == str(z["stats/xyz_gradient_accum"])
    assert rel(ours.xyz_gradient_accum, acc) < 1e-6
    ours.xyz_gradient_accum = acc
    # prune with a screen-size limit (all three criteria)
    ours.prune(0.0002, 0.005, extent, 20)
    assert ours._xyz.shape[0] < n1
    _assert_same_state(ours, z, "prune")
    # opacity reset: values, zeroed moments, kept step
    ours.reset_opacity()
    _assert_same_state(ours, z, "reset_opacity")
    # an optimizer step still works on the rebuilt parameters and matches torch.optim.Adam
    for n in PARAM_GROUPS:
        po = getattr(ours, _ATTR[n])
        po.grad = torch.randn(po.shape, device=DEV, generator=g) * 0.01
    ours.optimizer.step()
    for n in PARAM_GROUPS:
        e = util.relerr_sampled(getattr(ours, _ATTR[n]), z[f"adam/{n}_s"], z[f"adam/{n}_max"], DENSIFY_SAMPLE)
        assert e < 2e-6, (n, e)
    # split with nothing selected returns without touching anything (gaussian_model.py:507-508)
    before = ours._xyz.data_ptr()
    ours.densify_and_split(torch.zeros(ours._xyz.shape[0], 1, device=DEV), 1.0, extent)
    assert ours._xyz.data_ptr() == before


def test_training_loop_with_model_render_loss_and_densify(built_lib):
    """The pieces together the way train.py drives them: render -> fused loss -> backward -> stats -> densify/prune
    every few iterations -> Adam; checks that it runs, the loss goes down and the point count changes."""
    from s3gaussian_b200 import losses, synthetic as syn
    from s3gaussian_b200.gaussian_model import GaussianModel, default_optimization_params
    from s3gaussian_b200.gaussian_renderer import render, PipelineParams
    cloud = syn.make_cloud(30000, seed=3)
    cams = syn.waymo_ring(480, 320, frames=4)
    pc = GaussianModel(3).create_from_tensors(cloud.xyz.to(DEV), cloud.features_dc.to(DEV), cloud.features_rest.to(DEV),
                                              cloud.scaling.to(DEV), cloud.rotation.to(DEV), cloud.opacity.to(DEV))
    pc.active_sh_degree = 3
    pc.training_setup(default_optimization_params())
    bg = torch.zeros(3, device=DEV)
    pipe = PipelineParams()
    pipe.convert_SHs_python = False
    with torch.no_grad():
        targets = [(render(c, pc, pipe, bg, stage="coarse")["render"] * 0.5 + 0.25).clone() for c in cams[:3]]
        tdepth = [torch.full((1, 320, 480), 20.0, device=DEV) for _ in cams[:3]]
    first, last = {}, {}
    sizes = set()
    for it in range(1, 31):
        cam = (it - 1) % 3
        pc.update_learning_rate(it)
        out = render(cams[cam], pc, pipe, bg, stage="coarse")
        loss = losses.training_loss(out["render"], targets[cam], out["depth"], tdepth[cam])
        loss.backward()
        with torch.no_grad():
            pc.densification_step(out["viewspace_points"].grad, out["radii"])
            if it % 10 == 0:
                pc.densify(2e-6, 0.005, 30.0, None)
                pc.prune(2e-6, 0.005, 30.0, None)
            sizes.add(pc.get_xyz.shape[0])
        pc.optimizer.step()
        pc.optimizer.zero_grad(set_to_none=True)
        first.setdefault(cam, loss.item())
        last[cam] = loss.item()
    assert all(last[c] < first[c] for c in first), (first, last)
    assert len(sizes) > 1


# ---- checkpoints: the reference's capture() tuple (scene/gaussian_model.py:71-111) ----------------------------
def test_capture_restore_round_trip_with_reference_tuple(built_lib, tmp_path):
    """A checkpoint written the way train.py:531 does - torch.save((gaussians.capture(), iteration)) - by the
    REFERENCE's own capture()/training_setup() method bodies (ast-extracted from oracle/_ref, reference
    deform_network, torch.optim.Adam with two real steps) restores into our GaussianModel bit for bit, trains on,
    and our capture() restores into the reference's restore()."""
    import ast
    import os
    import ref_ext
    if not (ref_ext.gaussian_model_available() and ref_ext.deform_available()):
        pytest.skip("oracle/_ref/s3g_ref not present (run oracle/build_ref.sh)")
    from s3gaussian_b200 import synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    from s3gaussian_b200.gaussian_model import GaussianModel, default_optimization_params
    base = os.path.join(ref_ext.REF_DIR, "s3g_ref")
    ns = {"torch": torch, "nn": torch.nn, "np": np}
    for path, names in ((os.path.join(base, "utils", "general_utils.py"), {"get_expon_lr_func"}),
                        (os.path.join(base, "scene", "gaussian_model.py"),
                         {"capture", "restore", "training_setup", "get_xyz"})):
        for node in ast.walk(ast.parse(open(path).read())):
            if isinstance(node, ast.FunctionDef) and node.name in names:
                exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)

    class Ref:
        get_xyz = ns["get_xyz"]        # the extracted FunctionDef keeps its @property decorator
        capture, restore, training_setup = ns["capture"], ns["restore"], ns["training_setup"]
    ref_dn, _ = ref_ext.load_ref_deform()
    res, mres = (16, 12, 10, 7), (1, 2)
    args = ref_ext.ref_deform_args(res, mres)
    st = syn.make_deform_state(3, res, mres, aabb=((9.0, 4.0, 3.0), (-2.0, -4.0, -3.0)), weight_scale=0.2)
    P = 3000
    g = torch.Generator(device=DEV).manual_seed(5)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    ref = Ref()
    ref._deformation = ref_dn(args).to(DEV)
    ref._deformation.load_state_dict(st, strict=False)
    mk = lambda t: torch.nn.Parameter(t.requires_grad_(True))
    ref._xyz, ref._features_dc, ref._features_rest = mk(r(P, 3)), mk(r(P, 1, 3)), mk(r(P, 15, 3))
    ref._scaling, ref._rotation, ref._opacity = mk(r(P, 3)), mk(r(P, 4)), mk(r(P, 1))
    ref.active_sh_degree, ref.spatial_lr_scale = 2, 1.7
    ref._deformation_table = torch.ones(P, dtype=torch.bool, device=DEV)
    ref.max_radii2D = torch.rand(P, device=DEV, generator=g) * 30
    opt_args = default_optimization_params()
    ref.training_setup(opt_args)
    ref.xyz_gradient_accum = torch.rand(P, 1, device=DEV, generator=g)
    ref.denom = torch.randint(0, 5, (P, 1), device=DEV, generator=g).float()
    for _ in range(2):
        for grp in ref.optimizer.param_groups:
            for p in grp["params"]:
                p.grad = torch.randn(p.shape, device=DEV, generator=g) * 0.01
        ref.optimizer.step()
    path = str(tmp_path / "chkpnt_ref.pth")
    torch.save((ref.capture(), 1234), path)

    # ---- the reference checkpoint into our model ----
    model_args, it = torch.load(path, weights_only=False)
    assert it == 1234 and len(model_args) == 14
    ours = GaussianModel(3, deformation=deform_network(args))
    ours.restore(model_args, opt_args)
    assert ours.active_sh_degree == 2 and ours.spatial_lr_scale == 1.7
    for a in ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity", "max_radii2D",
              "xyz_gradient_accum", "denom", "_deformation_table"):
        assert torch.equal(getattr(ours, a).detach(), getattr(ref, a).detach()), a
    sd_o, sd_r = ours._deformation.state_dict(), ref._deformation.state_dict()
    assert set(sd_o) == set(sd_r)
    for k in sd_r:
        assert torch.equal(sd_o[k].to(DEV), sd_r[k]), k
    go, gr = ours.optimizer.param_groups, ref.optimizer.param_groups
    assert [x["name"] for x in go] == [x["name"] for x in gr]
    for a, b in zip(go, gr):
        assert a["lr"] == b["lr"] and len(a["params"]) == len(b["params"])
        for pa, pb in zip(a["params"], b["params"]):
            sa, sb = ours.optimizer.state[pa], ref.optimizer.state[pb]
            assert float(sa["step"]) == float(sb["step"]) == 2.0
            assert torch.equal(sa["exp_avg"].reshape(-1), sb["exp_avg"].reshape(-1)) or \
                torch.equal(sa["exp_avg"], sb["exp_avg"])
            assert torch.equal(sa["exp_avg_sq"], sb["exp_avg_sq"])
    # training resumes identically: one more step with the same gradients on both sides
    for a, b in zip(go, gr):
        for pa, pb in zip(a["params"], b["params"]):
            gt = torch.randn(pb.shape, device=DEV, generator=g) * 0.01
            pa.grad, pb.grad = gt.clone(), gt.clone()
    ours.optimizer.step()
    ref.optimizer.step()
    for a, b in zip(go, gr):
        for pa, pb in zip(a["params"], b["params"]):
            assert rel(pa, pb) < 2e-6, a["name"]

    # ---- our checkpoint into the reference's restore() ----
    path2 = str(tmp_path / "chkpnt_ours.pth")
    torch.save((ours.capture(), 1235), path2)
    model_args2, _ = torch.load(path2, weights_only=False)
    ref2 = Ref()
    ref2._deformation = ref_dn(args).to(DEV)
    ref2.restore(model_args2, opt_args)
    assert torch.equal(ref2._xyz.detach(), ours._xyz.detach()) and torch.equal(ref2.denom, ours.denom)
    for a, b in zip(ref2.optimizer.param_groups, ours.optimizer.param_groups):
        for pa, pb in zip(a["params"], b["params"]):
            assert float(ref2.optimizer.state[pa]["step"]) == 3.0
            assert torch.equal(ref2.optimizer.state[pa]["exp_avg_sq"], ours.optimizer.state[pb]["exp_avg_sq"])
