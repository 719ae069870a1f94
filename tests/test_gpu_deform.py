"""GPU parity of the fused HexPlane + decoder kernels and of render() (run with -m gpu).

Checkers: (1) tests/golden/deform_*.npz = outputs of the REAL reference deform_network;
(2) the torch restatement oracle/deform_oracle.py composed with the C rasterizer oracle for the
whole render(); (3) tests/golden/ref_*.npz = what the reference's own PyTorch module + CUDA extension
compute on the same GPU (tools/make_golden_refext.py).  Bars: 1e-4 relative on every output and gradient; the decoder runs 3xTF32."""
import os

import numpy as np
import pytest
import torch

import ref_ext
import util
from test_oracle_deform import GOLD, load_deform_case, rel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4
GOLD_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def build_net(z, st, flags):
    from s3gaussian_b200 import synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    net = deform_network(ref_ext.ref_deform_args([int(v) for v in z["resolution"]], [int(v) for v in z["multires"]], **flags))
    net.deformation_net.set_aabb(*[list(a) for a in syn.WAYMO_AABB])
    missing, unexpected = net.load_state_dict(st, strict=False)
    assert not unexpected
    return net.to(DEV)


@pytest.mark.parametrize("saved", [True, False], ids=["saved_activations", "recompute"])
@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[7:-4] for p in GOLD])
def test_fused_deform_matches_reference_golden(path, saved, built_lib, monkeypatch):
    """both backward variants against the reference's golden gradients: hidden activations kept by the tcgen05
    forward (s3g_deform_forward_save / s3g_deform_backward_saved) and recomputed in the backward kernel"""
    from s3gaussian_b200 import deformation
    monkeypatch.setattr(deformation, "SAVE_ACTIVATIONS", saved)
    z, st, flags = load_deform_case(path)
    net = build_net(z, st, flags)
    T = lambda k: torch.from_numpy(z[k]).to(DEV).requires_grad_(True)
    xyz, sc, ro, op, shs = T("in_xyz"), T("in_scales"), T("in_rot"), T("in_opacity"), T("in_shs")
    campos = torch.from_numpy(z["campos"]).to(DEV)
    outs = net.render_front(xyz, sc, ro, op, shs, float(z["time"]), campos, 3)
    names = ("out_means3D", "out_scales", "out_rot", "out_opacity", "out_colors", "out_dx", "out_dshs", "out_feat")
    for o, n in zip(outs, names):
        e = rel(o.detach().cpu().numpy().reshape(z[n].shape), z[n])
        assert e < TOL, (n, e)
    o_by = dict(zip(("m3", "sc", "ro", "op", "col", "dx", "dshs", "feat"), outs))
    ws = [torch.from_numpy(z[f"w{i}"]).to(DEV) for i in range(8)]
    loss = sum((o_by[k] * w.reshape(o_by[k].shape)).sum()
               for k, w in zip(("m3", "sc", "ro", "op", "col", "dx", "feat", "dshs"), ws))
    loss.backward()
    for leaf, n in zip((xyz, sc, ro, op, shs), ("g_xyz", "g_scales", "g_rot", "g_opacity", "g_shs")):
        assert rel(leaf.grad.cpu().numpy(), z[n]) < TOL, n
    checked = 0
    for k, p in net.named_parameters():
        key = "pg_" + k
        if p.grad is None:
            continue
        if key in z.files:
            assert rel(p.grad.cpu().numpy(), z[key]) < TOL, k
            checked += 1
        elif key + "_sample" in z.files:       # default-size planes: moments + strided sample
            gf = p.grad.reshape(-1).double()
            assert abs(float(gf.sum()) - float(z[key + "_sum"])) <= 2e-4 * float(z[key + "_abs"]) + 1e-12, k
            assert rel(p.grad.reshape(-1)[::997].cpu().numpy(), z[key + "_sample"]) < TOL, k
            checked += 1
    assert checked >= 28


@pytest.mark.parametrize("saved", [True, False], ids=["saved_activations", "recompute"])
@pytest.mark.parametrize("L", [1, 2, 3, 4])
def test_level_counts_against_the_oracle(L, saved, built_lib, monkeypatch):
    """1 .. 4 HexPlane levels (the level counts the kernels accept; feature widths 32 .. 128): the tcgen05 forward
    runs the feature layer as K-halves of 32+0, 64+0, 64+32 and 64+64 columns, the backward's generic-L
    instantiations cover 1 .. 3.  Forward
    outputs and every gradient against oracle/deform_oracle.py (float64 torch autograd), all heads enabled."""
    from oracle import deform_oracle as do
    from s3gaussian_b200 import deformation, synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    monkeypatch.setattr(deformation, "SAVE_ACTIVATIONS", saved)
    reso, multires = (12, 10, 8, 6), tuple(range(1, L + 1))
    aabb = ((9.0, 4.0, 3.0), (-2.0, -4.0, -3.0))
    flags = dict(no_ds=False, no_dr=False, no_do=False)
    st = syn.make_deform_state(5 + L, reso, multires, aabb=aabb, weight_scale=0.2)
    net = deform_network(ref_ext.ref_deform_args(reso, multires, **flags))
    net.deformation_net.set_aabb(list(aabb[0]), list(aabb[1]))
    missing, unexpected = net.load_state_dict(st, strict=False)
    assert not unexpected
    net = net.to(DEV)
    P = 333                                   # not a multiple of 64 / 128: ragged last tile
    g = torch.Generator().manual_seed(L)
    lo, hi = torch.tensor(aabb[1]), torch.tensor(aabb[0])
    xyz = lo + (hi - lo) * torch.rand(P, 3, generator=g)
    sc, ro, op = torch.randn(P, 3, generator=g) * 0.3 - 2, torch.randn(P, 4, generator=g), torch.randn(P, 1, generator=g)
    shs = torch.randn(P, 16, 3, generator=g) * 0.3
    campos = torch.tensor([0.3, -0.2, 6.0])
    t = 0.37
    ws = [torch.randn(*shape, generator=g) for shape in ((P, 3), (P, 3), (P, 4), (P, 1), (P, 3), (P, 3), (P, 16, 3), (P, 3))]
    # ours
    leaves = [v.clone().to(DEV).requires_grad_(True) for v in (xyz, sc, ro, op, shs)]
    outs = net.render_front(*leaves, t, campos.to(DEV), 3)
    sum((o * w.to(DEV)).sum() for o, w in zip(outs, ws)).backward()
    # oracle, float64
    std = {k: v.double().requires_grad_(v.is_floating_point() and "grid.aabb" not in k) for k, v in st.items()}
    ol = [v.clone().double().requires_grad_(True) for v in (xyz, sc, ro, op, shs)]
    d = do.deform_forward(std, ol[0], ol[1], ol[2], ol[3], ol[4], torch.full((P, 1), t, dtype=torch.float64),
                          no_dx=False, no_ds=False, no_dr=False, no_do=False, no_dshs=False, feat_head=True)
    front = do.render_front(ol[0], d, campos.double(), 3)
    ref_outs = (d["means3D"], front["scales"], front["rotations"], front["opacity"], front["colors_precomp"], d["dx"],
                d["dshs"], d["feat"])
    sum((o * w.double()).sum() for o, w in zip(ref_outs, ws)).backward()
    for o, r, n in zip(outs, ref_outs, ("means3D", "scales", "rot", "opacity", "colors", "dx", "dshs", "feat")):
        assert rel(o.detach().cpu().numpy(), r.detach().numpy().reshape(o.shape)) < TOL, (L, n)
    for a, b, n in zip(leaves, ol, ("xyz", "scales", "rot", "opacity", "shs")):
        assert rel(a.grad.cpu().numpy(), b.grad.numpy()) < TOL, (L, "d_" + n)
    checked = 0
    for k, p in net.named_parameters():
        if p.grad is None or k not in std or std[k].grad is None:
            continue
        assert rel(p.grad.cpu().numpy(), std[k].grad.numpy().reshape(p.shape)) < TOL, (L, k)
        checked += 1
    assert checked >= 6 * L + 20


def _small_fine_scene(P=400, W=80, H=48, seed=3):
    from s3gaussian_b200 import synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    from s3gaussian_b200.gaussian_renderer import GaussianModelLite
    cloud, cam = syn.make_small_scene(P=P, width=W, height=H, seed=seed)
    cam.time = 0.3
    st = syn.make_deform_state(seed, (16, 12, 10, 7), (1, 2, 4, 8), aabb=((9.0, 4.0, 3.0), (-2.0, -4.0, -3.0)), weight_scale=0.2)
    net = deform_network(ref_ext.ref_deform_args((16, 12, 10, 7), (1, 2, 4, 8)))
    net.deformation_net.set_aabb([9.0, 4.0, 3.0], [-2.0, -4.0, -3.0])
    net.load_state_dict(st, strict=False)
    pc = GaussianModelLite(cloud, net).to(DEV)
    return pc, cam, st, cloud


def test_render_fine_stage_matches_composed_oracles(built_lib, oracle_lib):
    """render(stage='fine', render_feat=True, return_dx=True): image, depth, feat image, dx, dshs and the
    gradients of a seeded loss w.r.t. xyz / shs / planes / MLP, against deform_oracle -> splat_oracle."""
    from oracle import deform_oracle as do
    from s3gaussian_b200.gaussian_renderer import render, PipelineParams
    pc, cam, st, cloud = _small_fine_scene()
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    out = render(cam, pc, PipelineParams(), bg, stage="fine", return_dx=True, render_feat=True)
    H, W = cam.image_height, cam.image_width
    g = torch.Generator().manual_seed(11)
    gc, gd, gf = torch.randn(3, H, W, generator=g), torch.randn(1, H, W, generator=g), torch.randn(3, H, W, generator=g)
    wdx, wds = torch.randn(cloud.P, 3, generator=g), torch.randn(cloud.P, 16, 3, generator=g)
    loss = (out["render"] * gc.to(DEV)).sum() + (out["depth"] * gd.to(DEV)).sum() + (out["feat"] * gf.to(DEV)).sum() + \
        (out["dx"] * wdx.to(DEV)).sum() + (out["dshs"] * wds.to(DEV)).sum()
    loss.backward()

    # ---- oracle composition (float64 deformation, float32 rasterizer) -----------------------
    state = {k: v.double().requires_grad_(k != "deformation_net.grid.aabb") for k, v in st.items()}
    xyz = cloud.xyz.double().requires_grad_(True)
    shs = cloud.get_features().double().requires_grad_(True)
    sc, ro, op = cloud.scaling.double().requires_grad_(True), cloud.rotation.double().requires_grad_(True), \
        cloud.opacity.double().requires_grad_(True)
    t = torch.full((cloud.P, 1), cam.time, dtype=torch.float64)
    d = do.deform_forward(state, xyz, sc, ro, op, shs, t)
    fr = do.render_front(xyz, d, cam.camera_center.double(), 3)

    def raster(colors):
        dd = dict(means3D=d["means3D"].detach().float(), opacities=fr["opacity"].detach().float(),
                  scales=fr["scales"].detach().float(), rotations=fr["rotations"].detach().float(), shs=None,
                  colors_precomp=colors.detach().float(), viewmatrix=cam.world_view_transform, projmatrix=cam.full_proj_transform,
                  campos=cam.camera_center, bg=bg.cpu(), W=W, H=H, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
                  sh_degree=3, cov3D_precomp=None)
        return dd
    o1 = util.oracle_run(oracle_lib, raster(fr["colors_precomp"]), gc, gd)
    o2 = util.oracle_run(oracle_lib, raster(d["feat"]), gf, torch.zeros(1, H, W))
    assert util.relerr(out["render"].detach().cpu().numpy(), o1["color"]) < TOL
    assert util.relerr(out["depth"].detach().cpu().numpy(), o1["depth"]) < TOL
    assert util.relerr(out["feat"].detach().cpu().numpy(), o2["color"]) < TOL
    assert np.array_equal(out["radii"].cpu().numpy(), o1["radii"])
    assert util.relerr(out["dx"].detach().cpu().numpy(), d["dx"].detach().numpy()) < TOL
    assert util.relerr(out["dshs"].detach().cpu().numpy(), d["dshs"].detach().numpy()) < TOL
    # chain the rasterizer-oracle gradients through the deformation oracle
    G = lambda o, k: torch.from_numpy(o["grads"][k]).double()
    torch.autograd.backward(
        [d["means3D"], fr["scales"], fr["rotations"], fr["opacity"], fr["colors_precomp"], d["feat"], d["dx"], d["dshs"]],
        [G(o1, "means3D") + G(o2, "means3D"), G(o1, "scales") + G(o2, "scales"), G(o1, "rotations") + G(o2, "rotations"),
         (G(o1, "opacity") + G(o2, "opacity")).reshape(-1, 1), G(o1, "colors"), G(o2, "colors"), wdx.double(), wds.double()])
    chk = [("xyz", pc._xyz.grad, xyz.grad), ("scaling", pc._scaling.grad, sc.grad), ("rotation", pc._rotation.grad, ro.grad),
           ("opacity", pc._opacity.grad, op.grad),
           ("features", torch.cat((pc._features_dc.grad, pc._features_rest.grad), 1), shs.grad)]
    for name, mine, ref in chk:
        assert util.relerr(mine.cpu().numpy(), ref.numpy()) < 5e-4, (name, util.relerr(mine.cpu().numpy(), ref.numpy()))
    sd = dict(pc._deformation.named_parameters())
    n = 0
    for k, v in state.items():
        if v.grad is not None and k in sd and sd[k].grad is not None:
            e = util.relerr(sd[k].grad.cpu().numpy(), v.grad.numpy())
            assert e < 5e-4, (k, e)
            n += 1
    assert n >= 28
    assert pc._xyz.grad.abs().max() > 0 and out["viewspace_points"].grad is not None


def test_render_coarse_stage_and_override_color(built_lib, oracle_lib):
    from s3gaussian_b200.gaussian_renderer import render, PipelineParams
    pc, cam, st, cloud = _small_fine_scene(P=300, seed=5)
    bg = torch.zeros(3, device=DEV)
    out = render(cam, pc, PipelineParams(), bg, stage="coarse")
    d = util.scene_inputs(cloud, cam, mode="sh", sh_degree=3, bg=(0, 0, 0))
    o = util.oracle_run(oracle_lib, d)
    assert util.relerr(out["render"].detach().cpu().numpy(), o["color"]) < TOL
    assert np.array_equal(out["radii"].cpu().numpy(), o["radii"])
    assert set(out) == {"render", "viewspace_points", "visibility_filter", "radii", "depth"}
    col = torch.rand(cloud.P, 3, device=DEV)
    out2 = render(cam, pc, PipelineParams(), bg, stage="coarse", override_color=col)
    d2 = dict(d); d2["shs"] = None; d2["colors_precomp"] = col.cpu()
    assert util.relerr(out2["render"].detach().cpu().numpy(), util.oracle_run(oracle_lib, d2)["color"]) < TOL
    out3 = render(cam, pc, PipelineParams(), bg, stage="fine", return_decomposition=True, return_dx=True)
    for k in ("render_d", "depth_d", "visibility_filter_d", "render_s", "depth_s", "visibility_filter_s", "dx", "dshs"):
        assert k in out3


STACK_CASES = [(200_000, 960, 640), (500_000, 1920, 1280)]
STACK_IDS = ["200k_960x640", "config3_500k_1920x1280"]
STACK_IMG, STACK_GRAD, STACK_PARAM = 1024, 512, 32      # stored values per image / Gaussian gradient / decoder gradient


def stack_case(P, W, H):
    """(cloud, camera, deformation state, dL/drender, dL/ddepth) of one reference-stack case"""
    from s3gaussian_b200 import synthetic as syn
    cloud = syn.make_cloud(P, seed=0, width=W, height=H)
    cam = syn.make_camera(W, H, (0, 0, 2.0), time=0.37)
    st = syn.make_deform_state(0, weight_scale=0.2)
    g = torch.Generator().manual_seed(2)
    gc, gd = torch.randn(3, H, W, generator=g).to(DEV), torch.randn(1, H, W, generator=g).to(DEV)
    return cloud, cam, st, gc, gd


def stack_loss(img, dep, feat, dx, dshs, gc, gd):
    return (img * gc).sum() + (dep * gd).sum() + feat.sum() * 0.1 + dx.abs().mean() + dshs.abs().mean()


@pytest.mark.parametrize("P,W,H", STACK_CASES, ids=STACK_IDS)
def test_render_matches_reference_stack_on_gpu(P, W, H, built_lib):
    """Same parameters through the REFERENCE stack on this GPU: its PyTorch deform_network + activations +
    eval_sh + its CUDA rasterizer (the code path of gaussian_renderer/__init__.py:89-166).  The second case is
    BASELINE config 3 at its real size (500k Gaussians, fine stage, 1920x1280, rgb + feat passes).  The reference's
    side is tests/golden/ref_render_stack.npz (tools/make_golden_refext.py): its images at STACK_IMG fixed pixels,
    its radii at fixed Gaussians, and its gradients at stored positions among their nonzero elements."""
    from s3gaussian_b200 import synthetic as syn
    from s3gaussian_b200.deformation import deform_network
    from s3gaussian_b200.gaussian_renderer import render, PipelineParams, GaussianModelLite
    z = util.load_golden(os.path.join(GOLD_DIR, "ref_render_stack.npz"))
    c = STACK_IDS[STACK_CASES.index((P, W, H))] + "/"
    cloud, cam, st, gc, gd = stack_case(P, W, H)
    args = ref_ext.ref_deform_args(syn.DEFAULT_RESOLUTION, syn.DEFAULT_MULTIRES)
    mine = deform_network(args); mine.deformation_net.set_aabb(*[list(a) for a in syn.WAYMO_AABB]); mine.load_state_dict(st, strict=False)
    util.fill_uncovered(mine, st)
    pc = GaussianModelLite(cloud, mine).to(DEV)
    bg = torch.zeros(3, device=DEV)
    out = render(cam.to(DEV), pc, PipelineParams(), bg, stage="fine", return_dx=True, render_feat=True)
    stack_loss(out["render"], out["depth"], out["feat"], out["dx"], out["dshs"], gc, gd).backward()
    # The two stacks feed the rasterizer means that differ in the last ulps (3xTF32 tensor-core decoder vs
    # cuBLAS fp32), so a handful of (pixel, Gaussian) pairs sit on the other side of the alpha >= 1/255 /
    # T >= 1e-4 thresholds (measured at 200k: 8e-6 of the pixels move by more than 1e-4, the largest by
    # 2.4e-3 = one near-threshold splat).  Bar: >= 99.99 % of the pixels within 1e-4 of the image range,
    # mean error < 1e-5, no pixel off by more than one splat's worth.
    def close_image(a, what):
        a, b = util.sample(a, STACK_IMG).astype(np.float64), z[c + what + "_s"].astype(np.float64)
        d = np.abs(a - b)
        scale = float(z[c + what + "_max"])
        assert float((d > 1e-4 * max(scale, 1.0)).mean()) < 1e-4, what
        assert float(d.mean()) < 1e-5 * max(scale, 1.0), what
        assert float(d.max()) < 2e-2 * max(scale, 1.0), what
    close_image(out["render"], "render")
    close_image(out["depth"], "depth")
    close_image(out["feat"], "feat")
    mism = int((util.sample(out["radii"], 4 * STACK_GRAD) != z[c + "radii_s"]).sum())
    assert mism <= max(2, P // 100000), mism      # deformed means differ in the last ulp (3xTF32 vs fp32 GEMM)
    # Gradients: the few threshold-flipped (pixel, Gaussian) pairs change those Gaussians' upstream gradients
    # by O(1), so element-wise max error is not meaningful across the two stacks; the relative L2 error is
    # (strict element-wise parity is what the golden and composed-oracle tests above establish).
    def rel_l2(t, key):
        a = t.detach().reshape(-1)[torch.from_numpy(z[key + "_idx"].astype(np.int64)).to(t.device)].double().cpu().numpy()
        b = z[key + "_s"].astype(np.float64)
        return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))
    assert rel_l2(pc._xyz.grad, c + "xyz") < 2e-2
    assert rel_l2(torch.cat((pc._features_dc.grad, pc._features_rest.grad), 1), c + "shs") < 2e-2
    names = str(z[c + "param_names"]).split()
    n = 0
    for k, p in pc._deformation.named_parameters():
        if p.grad is not None and k in names:
            assert rel_l2(p.grad, c + "p/" + k) < 2e-2, (k, rel_l2(p.grad, c + "p/" + k))
            n += 1
    assert n >= 28


@pytest.mark.parametrize("K,N", [(64, 64), (128, 64), (64, 48), (64, 16), (8, 16), (128, 32)])
def test_umma_selftest(K, N, built_lib):
    """tcgen05 building blocks (csrc/umma.cuh): a 128 x N x K GEMM issued as kind::tf32 UMMAs from
    canonical K-major smem operands into TMEM, read back with tcgen05.ld.  Single pass has tf32
    accuracy; the 3-pass split (what the decoder uses) has fp32 accuracy."""
    import ctypes as C
    from s3gaussian_b200 import _lib
    lib = _lib.load()
    g = torch.Generator(device=DEV).manual_seed(K * 131 + N)
    A = torch.randn(128, K, device=DEV, generator=g)
    B = torch.randn(N, K, device=DEV, generator=g)
    ref = A.double() @ B.double().t()
    for three, tol in ((0, 3e-3), (1, 2e-6)):
        D = torch.full((128, N), float("nan"), device=DEV)
        rc = lib.s3g_umma_selftest(A.data_ptr(), B.data_ptr(), D.data_ptr(), K, N, three,
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert rc == 0
        assert float((D.double() - ref).abs().max() / ref.abs().max()) < tol


COLD_SWITCH_FLAGS = dict(apply_rotation=True, no_ds=False, no_dr=False, no_do=False)
COLD_SWITCH_RESO, COLD_SWITCH_MRES = (16, 12, 10, 7), (1, 2, 4)
COLD_SWITCH_AABB = ((9.0, 4.0, 3.0), (-2.0, -4.0, -3.0))


def cold_switch_case(cls):
    """(network of class cls with the case's weights, cloud, camera) of the cold-switch render case"""
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=300, width=80, height=48, seed=3)
    cam.time = 0.3
    st = syn.make_deform_state(5, COLD_SWITCH_RESO, COLD_SWITCH_MRES, aabb=COLD_SWITCH_AABB, weight_scale=0.2)
    net = cls(ref_ext.ref_deform_args(COLD_SWITCH_RESO, COLD_SWITCH_MRES, **COLD_SWITCH_FLAGS))
    net.deformation_net.set_aabb(*[list(a) for a in COLD_SWITCH_AABB])
    net.load_state_dict(st, strict=False)
    return util.fill_uncovered(net, st), cloud, cam


def test_cold_switches_render_through_the_pytorch_path(built_lib):
    """apply_rotation (SURVEY section 8: "keep in PyTorch"): render(stage='fine') runs through
    deformation_cold.py + our rasterizer and equals the reference module's outputs fed to the same rasterizer
    (tests/golden/ref_cold_switch.npz: the reference module's dx in full, dshs at fixed positions)."""
    from s3gaussian_b200.deformation import deform_network
    from s3gaussian_b200.gaussian_renderer import render, PipelineParams, GaussianModelLite
    # (static_mlp / empty_voxel with random weights scatter the means off screen; their arithmetic is covered
    # on the CPU by tests/test_deform_cold_host.py - here the quaternion-product switch keeps a renderable scene)
    z = util.load_golden(os.path.join(GOLD_DIR, "ref_cold_switch.npz"))
    mine, cloud, cam = cold_switch_case(deform_network)
    assert "\n".join(sorted(mine.state_dict())) == str(z["keys"])
    pc = GaussianModelLite(cloud, mine).to(DEV)
    bg = torch.zeros(3, device=DEV)
    out = render(cam.to(DEV), pc, PipelineParams(), bg, stage="fine", return_dx=True, render_feat=True)
    (out["render"].sum() + out["feat"].sum() + out["depth"].sum()).backward()
    assert pc._xyz.grad is not None and float(pc._xyz.grad.abs().max()) > 0
    assert rel(out["dx"].detach().cpu().numpy(), z["dx"]) < 1e-5
    assert util.relerr_sampled(out["dshs"], z["dshs_s"], z["dshs_max"], 1024) < 1e-5
    assert out["render"].shape == (3, 48, 80) and torch.isfinite(out["render"]).all() and float(out["render"].max()) > 0
