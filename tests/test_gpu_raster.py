"""GPU parity tests of the rasterizer path (run with -m gpu on the B200 box).

Every call goes through the C ABI of libs3g_b200.so (via the drop-in Python
module).  Three checkers, in order of authority:
  1. tests/golden/raster_*.npz - outputs of the real reference extension;
  2. tests/golden/ref_*.npz - what the real reference extension computes at benchmark sizes, and the extension
     itself (oracle/_ref) where it was built;
  3. the CPU oracle (oracle/splat_oracle.c), pinned by (1) in test_oracle_golden.py.
Bars: bit-exact for radii / tiles_touched / sorted point_list / tile keys /
ranges / n_contrib; 1e-4 relative (of the tensor max) for colour, depth and all
gradients, as north_star states.
"""
import glob
import os

import numpy as np
import pytest
import torch

import ref_ext
import util
from test_oracle_golden import GOLD, load_case

pytestmark = pytest.mark.gpu

TOL = 1e-4
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ours(built_lib):
    from s3gaussian_b200 import diff_gaussian_rasterization as m
    return m


def check_state_vs(views, radii, R, ref_state):
    """ref_state: dict(num_rendered, radii, tiles_touched, point_list, keys(u64), ranges, n_contrib)"""
    assert R == int(ref_state["num_rendered"])
    np.testing.assert_array_equal(radii.cpu().numpy(), ref_state["radii"])
    np.testing.assert_array_equal(views["tiles_touched"], ref_state["tiles_touched"])
    np.testing.assert_array_equal(views["point_list"], ref_state["point_list"])
    np.testing.assert_array_equal(views["point_list_tiles"],
                                  (ref_state["keys"] >> np.uint64(32)).astype(np.uint32))
    np.testing.assert_array_equal(views["ranges"], ref_state["ranges"])
    np.testing.assert_array_equal(views["n_contrib"], ref_state["n_contrib"])


# --------------------------------------------------------------------- golden
@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[7:-4] for p in GOLD])
def test_cuda_matches_reference_golden(path, ours):
    z, d = load_case(path)
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    check_state_vs(views, radii, R, dict(num_rendered=z["num_rendered"], radii=z["radii"],
                                         tiles_touched=z["tiles_touched"], point_list=z["point_list"],
                                         keys=z["point_list_keys"], ranges=z["ranges"],
                                         n_contrib=z["n_contrib"]))
    vis = z["radii"] > 0
    # projected state: bit-exact against the reference (same expression trees, same FMA contraction)
    np.testing.assert_array_equal(views["xyAB"][vis, :2].view(np.uint32), z["means2D"][vis].view(np.uint32))
    conic = np.stack([views["xyAB"][:, 2], views["xyAB"][:, 3], views["Cod"][:, 0], views["Cod"][:, 1]], 1)
    np.testing.assert_array_equal(conic[vis].view(np.uint32), z["conic_opacity"][vis].view(np.uint32))
    np.testing.assert_array_equal(views["rgb"][vis, 3].view(np.uint32), z["depths"][vis].view(np.uint32))
    assert util.relerr(color.cpu().numpy(), z["color"]) < TOL
    assert util.relerr(depth.cpu().numpy(), z["depth"]) < TOL
    assert util.relerr(views["final_T"], z["final_T"]) < TOL
    # gradients
    gc, gd = torch.from_numpy(z["in_grad_color"]), torch.from_numpy(z["in_grad_depth"])
    out = util.run_module(ours, d, DEV, gc, gd)
    n = 0
    for k, g in out["grads"].items():
        key = "grad_" + k
        if key in z.files:
            assert util.relerr(g.cpu().numpy(), z[key]) < TOL, (k, util.relerr(g.cpu().numpy(), z[key]))
            n += 1
    assert n >= 5


# --------------------------------------------------------------------- oracle
@pytest.mark.parametrize("mode,deg,P,W,H,seed", [
    ("sh", 3, 400, 80, 64, 11), ("sh", 0, 257, 33, 17, 12), ("rgb", 0, 1000, 128, 96, 13),
    ("sh", 2, 64, 16, 16, 14), ("rgb", 0, 1, 40, 40, 15)])
def test_cuda_matches_cpu_oracle(mode, deg, P, W, H, seed, ours, oracle_lib):
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=P, width=W, height=H, seed=seed)
    d = util.scene_inputs(cloud, cam, mode=mode, sh_degree=deg)
    gc, gd = util.seeded_grads(d, seed)
    o = util.oracle_run(oracle_lib, d, gc, gd)
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    check_state_vs(views, radii, R, dict(num_rendered=o["R"], radii=o["radii"],
                                         tiles_touched=o["geometry"]["tiles_touched"],
                                         point_list=o["binning"]["point_list"], keys=o["binning"]["keys"],
                                         ranges=o["binning"]["ranges"], n_contrib=o["image"]["n_contrib"]))
    assert util.relerr(color.cpu().numpy(), o["color"]) < TOL
    assert util.relerr(depth.cpu().numpy(), o["depth"]) < TOL
    out = util.run_module(ours, d, DEV, gc, gd)
    names = {"means3D": "means3D", "means2D": "means2D", "opacities": "opacity", "scales": "scales",
             "rotations": "rotations", "shs": "sh", "colors_precomp": "colors"}
    for k, g in out["grads"].items():
        ref = o["grads"][names[k]].reshape(g.shape)
        if np.abs(ref).max() == 0:
            assert float(g.abs().max()) == 0
        else:
            assert util.relerr(g.cpu().numpy(), ref) < TOL, (k, util.relerr(g.cpu().numpy(), ref))


# ------------------------------------------------------------ real reference
GOLD_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NRUN = 4
IMG_SAMPLE, GRAD_SAMPLE = 1024, 512      # stored values per image / per gradient tensor of each benchmark-size case
BENCH_CASES = [(100_000, 960, 640, "sh", "front"), (100_000, 960, 640, "rgb", "front"),
               (500_000, 1920, 1280, "rgb", "front"), (500_000, 1920, 1280, "sh", "bench"),
               (2_000_000, 1920, 1280, "sh", "front"),
               (2_000_000, 1920, 1280, "sh", "bench"),
               # > 2.42 M points: the scan grid no longer fits resident at once and takes
               # the ticket + look-back path instead of the grid barrier
               (2_600_000, 1920, 1280, "rgb", "front")]


def bench_camera(W, H, rank=0):
    """the camera bench.py times on `rank` (bench.py: ring[1 + 3 * ((rank * 6) % 50)])"""
    from s3gaussian_b200 import synthetic as syn
    return syn.waymo_ring(W, H, frames=50)[1 + 3 * ((rank * 6) % 50)]


def bench_case_id(P, W, H, mode, view):
    return f"{P}_{W}x{H}_{mode}_{view}"


def bench_case_inputs(P, W, H, mode, view):
    from s3gaussian_b200 import synthetic as syn
    cloud = syn.make_cloud(P, seed=0)
    cam = syn.make_camera(W, H, (0, 0, 2.0)) if view == "front" else bench_camera(W, H, 0)
    d = util.scene_inputs(cloud, cam, mode=mode, sh_degree=3, bg=(0.0, 0.0, 0.0))
    gc, gd = util.seeded_grads(d, 7)
    return d, gc, gd


def scale_run_cases():
    """(rank, inputs) of the 7 other cameras of the 1->8 GPU scaling run, 2M Gaussians, 1920x1280"""
    from s3gaussian_b200 import synthetic as syn
    cloud = syn.make_cloud(2_000_000, seed=0)
    for rank in range(1, 8):
        yield rank, util.scene_inputs(cloud, bench_camera(1920, 1280, rank), mode="sh", sh_degree=3, bg=(0.0, 0.0, 0.0))


def check_state_record(views, radii, R, z, pre):
    """check_state_vs against a record of the reference's state (tools/make_golden_refext.py) under the key prefix `pre`"""
    assert R == int(z[pre + "num_rendered"])
    for k, v in (("radii", radii), ("tiles_touched", views["tiles_touched"]), ("point_list", views["point_list"]),
                 ("point_list_tiles", views["point_list_tiles"]), ("ranges", views["ranges"]),
                 ("n_contrib", views["n_contrib"])):
        assert util.digest(v) == str(z[pre + k]), k


@pytest.mark.parametrize("P,W,H,mode,view", BENCH_CASES)
def test_cuda_matches_reference_extension_at_benchmark_sizes(P, W, H, mode, view, ours):
    """BASELINE configs 2-4 geometry: identical Gaussians + camera through both implementations; integer state
    bit-exact, floats within 1e-4 of the tensor max AND element-wise within 1e-4 relative + a stated absolute
    floor.  view "bench" is the exact camera of the default bench.py line (waymo_ring[1]).  The reference's side is
    tests/golden/ref_raster_bench.npz (tools/make_golden_refext.py): digests of its integer state, its images at
    IMG_SAMPLE fixed pixels, its gradients (mean of NRUN runs) at GRAD_SAMPLE fixed positions among the visible
    Gaussians' rows, and each tensor's max and run-to-run spread."""
    z = util.load_golden(os.path.join(GOLD_DIR, "ref_raster_bench.npz"))
    c = bench_case_id(P, W, H, mode, view) + "/"
    d, gc, gd = bench_case_inputs(P, W, H, mode, view)
    # Both backward passes accumulate per-Gaussian gradients with unordered fp32 atomics, so two runs of the SAME
    # implementation differ: at 2.6 M the reference differs from itself by 1.3e-4 of the tensor max on the rotation
    # gradient of one needle-shaped Gaussian (tests/diag_grad_spread.py, profiles/r02q_grad_spread_2600k.log).  The
    # 1e-4 bar is therefore applied to the MEANS of NRUN runs of each (the accumulation noise averages out, a
    # systematic difference does not), and every single run must stay within 1e-4 + the reference's own spread.
    mine = [util.run_module(ours, d, DEV, gc, gd) for _ in range(NRUN)]
    m = mine[0]
    assert util.digest(m["radii"]) == str(z[c + "radii"])
    # forward images: 1e-4 of the max, and element-wise 1e-4 relative + 1e-6 absolute (colours are O(1), depths O(10))
    for k in ("color", "depth"):
        assert util.relerr_sampled(m[k], z[c + k + "_s"], z[c + k + "_max"], IMG_SAMPLE) < TOL, k
        frac, worst, _ = util.elementwise(util.sample(m[k], IMG_SAMPLE), z[c + k + "_s"], 1e-4, 1e-6)
        assert frac == 0.0, (k, frac, worst)
    # gradients at positions drawn among the rows of visible Gaussians (the radii just matched bit for bit); the
    # reference side is the mean of its NRUN runs, against which a single run of ours is no further than against one
    vis = m["radii"] > 0
    assert sorted(m["grads"]) == str(z[c + "grad_keys"]).split()
    for k in m["grads"]:
        g = c + "g/" + k
        M = [x["grads"][k].cpu().numpy() for x in mine]
        a, where = M[0], util.rows_mask(vis, M[0].shape)
        ref_s = z[g + "_mean_s"].astype(np.float64)
        assert ref_s.size == GRAD_SAMPLE
        tmax, spread = float(z[g + "_max"]), float(z[g + "_spread"])
        e_mean = util.relerr_sampled(np.mean(M, axis=0, dtype=np.float64), ref_s, tmax, GRAD_SAMPLE, where=where)
        e = util.relerr_sampled(a, ref_s, tmax, GRAD_SAMPLE, where=where)
        assert e_mean < TOL, (k, e_mean)
        assert e < TOL + spread / max(tmax, 1e-30), (k, e, spread / max(tmax, 1e-30))
        # element-wise: |ours - ref| <= 1e-4 |ref| + atol, atol = max(4 x the reference's own run-to-run spread
        # on this input, 1e-6 of the tensor max)
        atol = max(4.0 * spread, 1e-6 * tmax)
        frac, worst, idx = util.elementwise(util.sample(a, GRAD_SAMPLE, where=where), ref_s, 1e-4, atol)
        print(f"[elementwise] P={P} {mode} {view} {k}: max-normalised {e:.2e} (means of {NRUN} runs: {e_mean:.2e}), "
              f"atol {atol:.2e} (ref spread {spread:.2e}, tensor max {tmax:.2e}), "
              f"outside {frac:.2e}, worst ratio {worst:.2f}, nonzero samples {np.count_nonzero(ref_s)}")
        assert frac <= 1e-6, (k, frac, worst, idx)
    del mine
    # internal state bit for bit
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    check_state_record(views, radii, R, z, c)


def test_scale_run_cameras_integer_state_matches_reference(ours):
    """The 7 other cameras of the 1->8 GPU scaling run (rank r renders ring[1 + 3*((6r) % 50)]), 2M Gaussians,
    1920x1280: radii, num_rendered, sorted point_list, tile keys, ranges and n_contrib bit-exact against the
    reference extension, images within 1e-4 (tests/golden/ref_raster_scale_cams.npz)."""
    z = util.load_golden(os.path.join(GOLD_DIR, "ref_raster_scale_cams.npz"))
    for rank, d in scale_run_cases():
        c = f"rank{rank}/"
        color, radii, depth, R, views = util.ours_forward_state(d, DEV)
        check_state_record(views, radii, R, z, c)
        assert util.relerr_sampled(color, z[c + "color_s"], z[c + "color_max"]) < TOL, rank
        assert util.relerr_sampled(depth, z[c + "depth_s"], z[c + "depth_max"]) < TOL, rank


def test_mark_visible_matches_reference_and_oracle(ours, oracle_lib):
    from s3gaussian_b200 import synthetic as syn
    cloud = syn.make_cloud(50_000, seed=3)
    cam = syn.make_camera(640, 480, (0, 0, 2.0), yaw_deg=20)
    d = util.scene_inputs(cloud, cam, mode="rgb")
    mine = ours.GaussianRasterizer(util.settings_for(ours, d, DEV)).markVisible(d["means3D"].to(DEV))
    assert mine.dtype == torch.bool
    exp = oracle_lib.mark_visible(d["means3D"].numpy(), d["viewmatrix"].numpy())
    np.testing.assert_array_equal(mine.cpu().numpy(), exp)
    if ref_ext.available():
        ref = ref_ext.load()
        theirs = ref.GaussianRasterizer(util.settings_for(ref, d, DEV)).markVisible(d["means3D"].to(DEV))
        assert torch.equal(mine, theirs)


# ------------------------------------------------------------ edge cases
def test_empty_cloud_and_all_culled(ours):
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=8, width=40, height=24, seed=2)
    d = util.scene_inputs(cloud, cam, mode="rgb")
    # P == 0: outputs stay zero like the reference glue (rasterize_points.cu:82)
    d0 = dict(d)
    for k in ("means3D", "opacities", "scales", "rotations", "colors_precomp"):
        d0[k] = d[k][:0]
    out = util.run_module(ours, d0, DEV)
    assert out["radii"].numel() == 0 and float(out["color"].abs().max()) == 0
    # everything behind the camera: R == 0, colour == background, depth == 0, zero grads
    d1 = dict(d)
    d1["means3D"] = d["means3D"].clone()
    d1["means3D"][:, 0] = -5.0
    gc, gd = util.seeded_grads(d1, 3)
    out = util.run_module(ours, d1, DEV, gc, gd)
    assert int((out["radii"] > 0).sum()) == 0
    bg = d1["bg"].view(3, 1, 1).to(DEV)
    assert torch.equal(out["color"], bg.expand_as(out["color"]).contiguous())
    assert float(out["depth"].abs().max()) == 0
    for k, g in out["grads"].items():
        assert float(g.abs().max()) == 0, k


def test_huge_gaussian_covers_every_tile(ours, oracle_lib):
    """one splat whose rect is the whole grid (cooperative emission path) + small ones"""
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=40, width=200, height=120, seed=9)
    cloud.scaling[0] = 2.0          # exp(2) m: fills the screen
    cloud.xyz[0] = torch.tensor([6.0, 0.0, 0.0])
    d = util.scene_inputs(cloud, cam, mode="sh", sh_degree=1)
    gc, gd = util.seeded_grads(d, 4)
    o = util.oracle_run(oracle_lib, d, gc, gd)
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    assert views["tiles_touched"][0] == 13 * 8
    check_state_vs(views, radii, R, dict(num_rendered=o["R"], radii=o["radii"],
                                         tiles_touched=o["geometry"]["tiles_touched"],
                                         point_list=o["binning"]["point_list"], keys=o["binning"]["keys"],
                                         ranges=o["binning"]["ranges"], n_contrib=o["image"]["n_contrib"]))
    assert util.relerr(color.cpu().numpy(), o["color"]) < TOL


def test_extreme_opacity_and_anisotropy(ours, oracle_lib):
    """opacity below 1/255 (never blends), opacity ~1 (alpha clamps at 0.99), needle-shaped
    splats (cull threshold falls back to 'never cull')"""
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=300, width=96, height=64, seed=21)
    cloud.opacity[:60] = -8.0        # sigmoid ~ 3e-4 < 1/255
    cloud.opacity[60:120] = 12.0     # ~ 1.0
    cloud.scaling[120:180, 0] += 3.0  # needles
    cloud.scaling[120:180, 1] -= 2.0
    d = util.scene_inputs(cloud, cam, mode="rgb")
    gc, gd = util.seeded_grads(d, 5)
    o = util.oracle_run(oracle_lib, d, gc, gd)
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    check_state_vs(views, radii, R, dict(num_rendered=o["R"], radii=o["radii"],
                                         tiles_touched=o["geometry"]["tiles_touched"],
                                         point_list=o["binning"]["point_list"], keys=o["binning"]["keys"],
                                         ranges=o["binning"]["ranges"], n_contrib=o["image"]["n_contrib"]))
    assert util.relerr(color.cpu().numpy(), o["color"]) < TOL
    # In this regime (alpha clamped at 0.99, T divided by 0.01 per layer) the gradients are
    # ill-conditioned: the reference itself moves by ~2e-3 between runs (unordered fp32
    # atomics, backward.cu:550-587) and sits ~2e-3..6e-3 from the double-accumulating oracle,
    # so the bar here is 2e-2 against the oracle and "as close as the reference is to itself"
    # against the reference extension.
    out = util.run_module(ours, d, DEV, gc, gd)
    names = {"means3D": "means3D", "opacities": "opacity", "scales": "scales", "rotations": "rotations",
             "colors_precomp": "colors", "means2D": "means2D"}
    for k, ok in names.items():
        e = util.relerr(out["grads"][k].cpu().numpy(), o["grads"][ok].reshape(out["grads"][k].shape))
        assert e < 2e-2, (k, e)
    if ref_ext.available():
        ref = ref_ext.load()
        # the reference's spread is itself a random sample (two runs can happen to agree to 3e-4 or differ by 3e-3),
        # so it is taken as the largest of four runs against the first, with a floor of 1e-2 = 5 x its typical value
        runs = [util.run_module(ref, d, DEV, gc, gd) for _ in range(5)]
        for k in names:
            r0 = runs[0]["grads"][k].cpu().numpy()
            noise = max(util.relerr(r["grads"][k].cpu().numpy(), r0) for r in runs[1:])
            e = util.relerr(out["grads"][k].cpu().numpy(), r0)
            assert e < max(5 * noise, 1e-2), (k, e, noise)


# ------------------------------------------- size-independent properties, full size
def test_full_size_properties(ours):
    """2M Gaussians, 1920x1280 (BASELINE metric size): sortedness, range consistency,
    checksum of counts, determinism of the forward, linearity of the backward."""
    from s3gaussian_b200 import synthetic as syn
    P, W, H = 2_000_000, 1920, 1280
    cloud = syn.make_cloud(P, seed=0)
    cam = syn.make_camera(W, H, (0, 0, 2.0))
    d = util.scene_inputs(cloud, cam, mode="rgb", bg=(0.0, 0.0, 0.0))
    color, radii, depth, R, v = util.ours_forward_state(d, DEV)
    tt, pl, plt, rng = v["tiles_touched"], v["point_list"], v["point_list_tiles"], v["ranges"]
    assert int(tt.astype(np.int64).sum()) == R                       # checksum of counts
    assert np.array_equal((tt > 0), radii.cpu().numpy() > 0)
    assert np.all(np.diff(plt.astype(np.int64)) >= 0)                 # sorted by tile
    depth_bits = v["rgb"][:, 3].view(np.uint32)[pl].astype(np.int64)
    key = (plt.astype(np.int64) << 32) | depth_bits
    assert np.all(np.diff(key) >= 0)                                  # then by depth bits
    ties = np.diff(key) == 0
    assert np.all(np.diff(pl.astype(np.int64))[ties] > 0)             # stable: ties keep index order
    counts = np.bincount(plt, minlength=rng.shape[0])
    lens = (rng[:, 1].astype(np.int64) - rng[:, 0].astype(np.int64))
    assert np.array_equal(lens, counts)                               # ranges == histogram
    nz = counts > 0
    assert np.array_equal(rng[nz, 0], (np.cumsum(counts) - counts)[nz].astype(np.uint32))
    assert np.all(rng[~nz] == 0)
    assert np.all(v["n_contrib"].reshape(H, W) <= lens.reshape(80, 120).repeat(16, 0).repeat(16, 1))
    # determinism of the forward (bitwise)
    color2, radii2, depth2, R2, v2 = util.ours_forward_state(d, DEV)
    assert R2 == R and torch.equal(color, color2) and torch.equal(depth, depth2)
    assert np.array_equal(v2["point_list"], pl)
    # linearity of the backward in dL/dout
    g1c, g1d = util.seeded_grads(d, 1)
    g2c, g2d = util.seeded_grads(d, 2)
    a = util.run_module(ours, d, DEV, g1c, g1d)["grads"]
    b = util.run_module(ours, d, DEV, g2c, g2d)["grads"]
    c = util.run_module(ours, d, DEV, g1c + 2 * g2c, g1d + 2 * g2d)["grads"]
    for k in a:
        lin = (a[k].double() + 2 * b[k].double())
        e = float((c[k].double() - lin).abs().max() / (lin.abs().max() + 1e-30))
        assert e < 5e-4, (k, e)


def test_radix_sort_standalone(built_lib):
    """the hand-written onesweep sort vs torch.sort(stable=True), incl. ragged sizes"""
    import ctypes as C
    from s3gaussian_b200 import _lib
    lib = built_lib
    g = torch.Generator(device=DEV).manual_seed(0)
    for n, b0, b1, hi in [(1, 0, 32, 2**31), (33, 0, 8, 200), (4096, 0, 32, 2**31), (4097, 0, 14, 9600),
                          (123_457, 3, 17, 2**20), (1_000_003, 0, 14, 9600), (2_000_000, 0, 32, 2**31)]:
        keys = torch.randint(0, hi, (n,), device=DEV, generator=g, dtype=torch.int64).to(torch.int32)
        vals = torch.arange(n, device=DEV, dtype=torch.int32)
        ko, vo = torch.empty_like(keys), torch.empty_like(vals)
        tmp = torch.empty(lib.s3g_sort_temp_bytes(n), dtype=torch.uint8, device=DEV)
        kin, vin = keys.clone(), vals.clone()
        _lib.check(lib.s3g_sort_pairs_u32(n, kin.data_ptr(), vin.data_ptr(), ko.data_ptr(), vo.data_ptr(), b0, b1,
                                          tmp.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "sort")
        torch.cuda.synchronize()
        dig = (keys.to(torch.int64) >> b0) & ((1 << (b1 - b0)) - 1)
        _, perm = torch.sort(dig, stable=True)
        assert torch.equal(vo.to(torch.int64), perm), (n, b0, b1)
        assert torch.equal(ko, keys[perm])


def test_binning_capacity_overflow_is_repeated_not_truncated(ours, oracle_lib):
    """The forward enqueues the binning against the capacity remembered from the previous call on this thread and
    checks the true instance count afterwards; a call whose count outgrew it must come out identical to a fresh
    one (the tail is repeated with a larger arena), and a much smaller call after a big one must not see stale
    state."""
    from s3gaussian_b200 import synthetic as syn
    small_cloud, small_cam = syn.make_small_scene(P=50, width=64, height=48, seed=31)
    big_cloud, big_cam = syn.make_small_scene(P=6000, width=320, height=208, seed=32)
    ds = util.scene_inputs(small_cloud, small_cam, mode="rgb")
    db = util.scene_inputs(big_cloud, big_cam, mode="sh", sh_degree=2)
    ob, os_ = util.oracle_run(oracle_lib, db), util.oracle_run(oracle_lib, ds)
    assert ob["R"] > 20 * max(os_["R"], 1)
    for d, o in ((ds, os_), (db, ob), (ds, os_), (db, ob)):
        color, radii, depth, R, views = util.ours_forward_state(d, DEV)
        check_state_vs(views, radii, R, dict(num_rendered=o["R"], radii=o["radii"],
                                             tiles_touched=o["geometry"]["tiles_touched"],
                                             point_list=o["binning"]["point_list"], keys=o["binning"]["keys"],
                                             ranges=o["binning"]["ranges"], n_contrib=o["image"]["n_contrib"]))
        assert util.relerr(color.cpu().numpy(), o["color"]) < TOL
        assert util.relerr(depth.cpu().numpy(), o["depth"]) < TOL


def test_shared_binning_two_colour_sets_equal_two_passes(ours):
    """forward_aux / s3g_rasterize_*_aux: colour image + feature image composited on one preprocess + sort must equal
    two full passes (what gaussian_renderer/__init__.py:173-186 does) - images, and the gradients of the SUM of both
    losses w.r.t. geometry, opacity and both colour sets; against our own two passes and the reference's."""
    from s3gaussian_b200 import synthetic as syn
    P, W, H = 60_000, 640, 416
    cloud = syn.make_cloud(P, seed=4, width=W, height=H)
    cam = syn.make_camera(W, H, (0, 0, 2.0))
    d = util.scene_inputs(cloud, cam, mode="rgb", bg=(0.3, 0.1, 0.2))
    g = torch.Generator().manual_seed(8)
    feat = torch.rand(P, 3, generator=g)
    gc, gd = util.seeded_grads(d, 21)
    gf = torch.randn(3, H, W, generator=g)

    def run(mod, fused):
        t = {k: d[k].to(DEV).clone().requires_grad_(True) for k in ("means3D", "opacities", "scales", "rotations", "colors_precomp")}
        fa = feat.to(DEV).clone().requires_grad_(True)
        m2d = torch.zeros_like(t["means3D"], requires_grad=True)
        rast = mod.GaussianRasterizer(util.settings_for(mod, d, DEV))
        kw = dict(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"], scales=t["scales"], rotations=t["rotations"])
        if fused:
            color, radii, depth, aux = rast.forward_aux(colors_aux=fa, colors_precomp=t["colors_precomp"], **kw)
        else:
            color, radii, depth = rast(colors_precomp=t["colors_precomp"], **kw)
            aux, _, _ = rast(colors_precomp=fa, **kw)
        ((color * gc.to(DEV)).sum() + (depth * gd.to(DEV)).sum() + (aux * gf.to(DEV)).sum()).backward()
        grads = {k: v.grad.detach() for k, v in t.items()}
        grads["colors_aux"], grads["means2D"] = fa.grad.detach(), m2d.grad.detach()
        return color.detach(), depth.detach(), aux.detach(), radii, grads
    c1, d1, a1, r1, g1 = run(ours, True)
    c2, d2, a2, r2, g2 = run(ours, False)
    assert torch.equal(r1, r2) and torch.equal(c1, c2) and torch.equal(d1, d2)
    assert util.relerr(a1.cpu().numpy(), a2.cpu().numpy()) < 1e-6
    for k in g2:
        e = util.relerr(g1[k].cpu().numpy(), g2[k].cpu().numpy())
        assert e < 2e-5, (k, e)
    if ref_ext.available():
        c3, d3, a3, r3, g3 = run(ref_ext.load(), False)
        assert torch.equal(r1, r3)
        assert util.relerr(a1.cpu().numpy(), a3.cpu().numpy()) < TOL
        for k in g3:
            e = util.relerr(g1[k].cpu().numpy(), g3[k].cpu().numpy())
            assert e < TOL, (k, e)


def test_more_than_16k_tiles_uses_the_global_histogram_path(ours, oracle_lib):
    """2576x1664 = 161 x 104 = 16 744 tiles: the tile histogram no longer fits the emit kernel's shared-memory table
    (emit_instances_kernel<false>, direct global atomics) and the tile ids need 15 key bits."""
    from s3gaussian_b200 import synthetic as syn
    cloud, cam = syn.make_small_scene(P=2500, width=2576, height=1664, seed=41)
    d = util.scene_inputs(cloud, cam, mode="rgb")
    o = util.oracle_run(oracle_lib, d)
    color, radii, depth, R, views = util.ours_forward_state(d, DEV)
    assert views["ranges"].shape[0] == 161 * 104
    # 4.3 M pixels x ~450 list entries: the CPU oracle's expf (glibc) and CUDA's differ in the last bit often enough
    # for a handful of alpha >= 1/255 decisions to flip, so n_contrib is compared bit for bit against the REFERENCE
    # EXTENSION (same device arithmetic) and only approximately against the oracle
    nc = views["n_contrib"].copy()
    check_state_vs(dict(views, n_contrib=o["image"]["n_contrib"]), radii, R,
                   dict(num_rendered=o["R"], radii=o["radii"], tiles_touched=o["geometry"]["tiles_touched"],
                        point_list=o["binning"]["point_list"], keys=o["binning"]["keys"],
                        ranges=o["binning"]["ranges"], n_contrib=o["image"]["n_contrib"]))
    assert int((nc != o["image"]["n_contrib"]).sum()) <= 8
    cerr = np.abs(color.cpu().numpy() - o["color"]).max(0)               # a flipped pixel differs by one splat's worth
    assert int((cerr > TOL * np.abs(o["color"]).max()).sum()) <= 64 and float(cerr.mean()) < 1e-6    # of 4.3 M pixels
    if ref_ext.available():
        ref = ref_ext.load()
        E = torch.Tensor([])
        g = lambda k: d[k].to(DEV).contiguous() if d[k] is not None else E
        R0, rc, rdep, rrad, gb, bb, ib = ref._C.rasterize_gaussians(
            d["bg"].to(DEV), g("means3D"), g("colors_precomp"), g("opacities"), g("scales"), g("rotations"), 1.0,
            g("cov3D_precomp"), d["viewmatrix"].to(DEV), d["projmatrix"].to(DEV), d["tanfovx"], d["tanfovy"], d["H"], d["W"],
            g("shs"), d["sh_degree"], d["campos"].to(DEV), False, False)
        torch.cuda.synchronize()
        ri = ref_ext.decode_image(ib, d["W"] * d["H"])
        assert R0 == R
        np.testing.assert_array_equal(nc, ri["n_contrib"])
        assert util.relerr(color.cpu().numpy(), rc.cpu().numpy()) < TOL
