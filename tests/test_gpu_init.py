"""GPU parity of the initialisation path (run with -m gpu): distCUDA2 against (1) the goldens of the real
reference extension, (2) the brute-force oracle, (3) the goldens of the reference extension at benchmark size;
create_from_pcd and the .ply round trip through the model."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_golden_knn as mk                                     # noqa: E402
import util                                                      # noqa: E402
from test_init_io import KNN_GOLD                                # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("path", KNN_GOLD, ids=[os.path.basename(p)[4:-4] for p in KNN_GOLD])
def test_distcuda2_matches_reference_golden(path, built_lib):
    from s3gaussian_b200.simple_knn import distCUDA2
    z = np.load(path)
    pts = mk.knn_inputs(str(z["name"]), int(z["P"]), int(z["seed"]))
    ours = distCUDA2(pts.to(DEV)).cpu().numpy()
    ref = z["mean_dist2"]
    fin = np.isfinite(ref)
    assert np.array_equal(fin, np.isfinite(ours))
    assert np.array_equal(ours[fin], ref[fin])                   # same arithmetic: bit-exact


def knn_ext_cases():
    """(name, points) compared with the reference extension at benchmark size (tests/golden/ref_knn_ext.npz)"""
    return [("clustered_2M", mk.knn_inputs("clustered", 2_000_000, 12)),
            ("uniform_500k", mk.knn_inputs("uniform", 500_000, 13)), ("one_point", torch.zeros(1, 3))]


def test_distcuda2_matches_oracle_and_reference_extension(built_lib):
    from oracle import knn_oracle
    from s3gaussian_b200.simple_knn import distCUDA2
    pts = mk.knn_inputs("clustered", 20000, 11)
    ours = distCUDA2(pts.to(DEV)).cpu().numpy()
    assert np.allclose(ours, knn_oracle.mean_dist2(pts.numpy()), rtol=2e-6, atol=1e-12)
    # the reference extension's results, bit for bit (tools/make_golden_refext.py)
    z = util.load_golden(os.path.join(ROOT, "tests", "golden", "ref_knn_ext.npz"))
    for name, p in knn_ext_cases():
        assert util.digest(distCUDA2(p.to(DEV))) == str(z[name]), name
    assert distCUDA2(torch.zeros(0, 3, device=DEV)).shape == (0,)
    assert torch.isinf(distCUDA2(torch.zeros(1, 3, device=DEV))).all()


def test_create_from_pcd_and_ply_round_trip(built_lib, tmp_path):
    from types import SimpleNamespace
    from s3gaussian_b200.gaussian_model import GaussianModel
    from s3gaussian_b200.simple_knn import distCUDA2
    g = torch.Generator().manual_seed(2)
    pts = (torch.rand(5000, 3, generator=g) * 30).numpy()
    cols = torch.rand(5000, 3, generator=g).numpy()
    m = GaussianModel(3).create_from_pcd(SimpleNamespace(points=pts, colors=cols), 7.5)
    assert m.spatial_lr_scale == 7.5 and m._xyz.shape == (5000, 3) and m._features_rest.shape == (5000, 15, 3)
    d2 = torch.clamp_min(distCUDA2(torch.from_numpy(pts).to(DEV)), 1e-7)
    assert torch.equal(m._scaling.data, torch.log(torch.sqrt(d2))[:, None].repeat(1, 3))
    assert torch.allclose(m.get_opacity, torch.full((5000, 1), 0.1, device=DEV), atol=1e-6)
    assert torch.allclose(m._features_dc[:, 0] * 0.28209479177387814 + 0.5, torch.from_numpy(cols).to(DEV), atol=1e-6)
    assert float(m._features_rest.detach().abs().max()) == 0.0 and torch.equal(m._rotation.data[:, 0], torch.ones(5000, device=DEV))
    path = str(tmp_path / "pc" / "point_cloud.ply")
    m.save_ply(path)
    n = GaussianModel(3).load_ply(path)
    for a in ("_xyz", "_features_dc", "_features_rest", "_opacity", "_scaling", "_rotation"):
        assert torch.equal(getattr(n, a).data, getattr(m, a).data), a
    assert n.active_sh_degree == 3
