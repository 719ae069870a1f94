"""Host-side (CPU) checks of GaussianModel against the reference's own method bodies: learning-rate schedule
(scene/gaussian_model.py:203-218), taken from oracle/_ref with ast and executed unmodified by
tools/make_golden_refext.py; its results are tests/golden/ref_lr_schedule.npz."""
import os
from argparse import Namespace

import numpy as np
import torch
import torch.nn as nn

import util


GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ITERATIONS = (1, 2, 500, 7000, 19999, 20000, 30000)

OPT = Namespace(percent_dense=0.01, position_lr_init=0.00016, position_lr_final=0.0000016, position_lr_delay_mult=0.01,
                position_lr_max_steps=20000, deformation_lr_init=0.000016, deformation_lr_final=0.0000016,
                deformation_lr_delay_mult=0.01, grid_lr_init=0.0016, grid_lr_final=0.000016, feature_lr=0.0025,
                opacity_lr=0.05, scaling_lr=0.005, rotation_lr=0.001)   # arguments/__init__.py:236-262


class _Deform(nn.Module):
    def __init__(self):
        super().__init__()
        self.mlp = nn.Linear(4, 4)
        self.grid = nn.Parameter(torch.zeros(1, 2, 3, 3))

    def get_mlp_parameters(self):
        return list(self.mlp.parameters())

    def get_grid_parameters(self):
        return [self.grid]


def _our_model():
    from s3gaussian_b200.gaussian_model import GaussianModel
    m = GaussianModel(3, deformation=_Deform())
    mk = lambda *s: nn.Parameter(torch.zeros(*s))
    m._xyz, m._features_dc, m._features_rest = mk(5, 3), mk(5, 1, 3), mk(5, 15, 3)
    m._scaling, m._rotation, m._opacity = mk(5, 3), mk(5, 4), mk(5, 1)
    m.spatial_lr_scale = 3.7
    m.training_setup(OPT)
    return m


def test_learning_rates_follow_the_reference_schedule():
    """tests/golden/ref_lr_schedule.npz: the reference's update_learning_rate over the same groups
    (tools/make_golden_refext.py)."""
    z = util.load_golden(os.path.join(GOLD, "ref_lr_schedule.npz"))
    m = _our_model()
    s = m.spatial_lr_scale
    names = [g["name"] for g in m.optimizer.param_groups]
    assert names == ["xyz", "deformation", "grid", "f_dc", "f_rest", "opacity", "scaling", "rotation"]
    assert names == list(z["group_names"]) and tuple(z["iterations"]) == ITERATIONS
    for i, it in enumerate(ITERATIONS):
        lr_ours = m.update_learning_rate(it)
        assert lr_ours == z["lr"][i]
        for go, lr_ref in zip(m.optimizer.param_groups, z["group_lr"][i]):
            assert go["lr"] == lr_ref, (it, go["name"])
    d = {g["name"]: g["lr"] for g in m.optimizer.param_groups}
    assert abs(d["deformation"] - OPT.deformation_lr_final * s) < 1e-12      # decayed 1.6e-5 -> 1.6e-6 (x scale)


def test_zero_width_feature_rows_survive_row_surgery_plan():
    """max_sh_degree == 0 gives _features_rest [P,0,3]: the row-gather descriptor list must skip it
    (s3g_gather_rows rejects row_floats <= 0)."""
    import inspect
    from s3gaussian_b200.gaussian_model import GaussianModel
    src = inspect.getsource(GaussianModel._rebuild)
    assert "rf == 0" in src
