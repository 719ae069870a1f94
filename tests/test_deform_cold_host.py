"""CPU: the PyTorch cold path of the deformation module (s3gaussian_b200/deformation_cold.py: static_mlp, empty_voxel,
apply_rotation - the switches SURVEY section 8 keeps out of the CUDA kernels) against the REAL reference module on the
same state_dict: outputs, input gradients and parameter gradients.  The reference's results are
tests/golden/ref_deform_cold.npz (tools/make_golden_refext.py).  On one machine the two agree bit for bit; across
machines CPU torch does not (its kernels differ by instruction set: 6e-7 of the tensor max measured between the AVX-512
and the unvectorised build of the same run), so the stored results are matched to TOL of each tensor's max.  The product
guards these paths to CUDA tensors like everything else; the arithmetic itself is device-independent torch and is
checked here."""
import os

import numpy as np
import pytest
import torch

import ref_ext
import util

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = [dict(static_mlp=True, no_ds=False, no_dr=False, no_do=False),
         dict(empty_voxel=True, no_ds=False, no_do=False),
         dict(apply_rotation=True, no_dr=False),
         dict(static_mlp=True, apply_rotation=True, no_dr=False, no_dshs=True, feat_head=False)]
IDS = ["static_mlp", "empty_voxel", "apply_rotation", "mixed"]
RESO, MRES = (16, 12, 10, 7), (1, 2, 4)
P = 150
TOL = 1e-5


def make_net(cls, flags):
    """One case's network (reference or ours): the seeded HexPlane + decoder state, and the parameters that state does
    not cover (time net, static_mlp) drawn from a generator of their own in name order."""
    from s3gaussian_b200 import synthetic as syn
    st = syn.make_deform_state(3, RESO, MRES, weight_scale=0.2)
    net = cls(ref_ext.ref_deform_args(RESO, MRES, **flags))
    net.deformation_net.set_aabb(*[list(a) for a in syn.WAYMO_AABB])
    net.load_state_dict(st, strict=False)
    return util.fill_uncovered(net, st)


def case_inputs(flags, net):
    """(inputs, f(outputs) -> output weights of the scalar loss) of one case, from one seeded generator."""
    from s3gaussian_b200 import synthetic as syn
    g = torch.Generator().manual_seed(4)
    if flags.get("empty_voxel"):
        net.deformation_net.empty_voxel.grid.data.copy_(torch.rand(1, 1, 64, 64, 64, generator=g))
    lo, hi = torch.tensor(syn.WAYMO_AABB[1]), torch.tensor(syn.WAYMO_AABB[0])
    base = [lo + (hi - lo) * torch.rand(P, 3, generator=g), torch.randn(P, 3, generator=g), torch.randn(P, 4, generator=g),
            torch.randn(P, 1, generator=g), torch.randn(P, 16, 3, generator=g)]
    return base, lambda outs: [None if x is None else torch.randn(x.shape, generator=g) for x in outs]


@pytest.mark.parametrize("flags", CASES, ids=IDS)
def test_cold_path_equals_reference_module(flags):
    from s3gaussian_b200 import deformation_cold as dc
    from s3gaussian_b200.deformation import deform_network
    z = util.load_golden(os.path.join(GOLD, "ref_deform_cold.npz"))
    cid = IDS[CASES.index(flags)]
    ours = make_net(deform_network, flags)
    assert ours.deformation_net.cold
    assert "\n".join(sorted(ours.state_dict())) == str(z[f"{cid}/keys"])      # incl. static_mlp / empty_voxel.grid
    base, weights = case_inputs(flags, ours)
    b_in = [t.clone().requires_grad_(True) for t in base]
    b = dc.forward_dynamic(ours.deformation_net, *b_in, 0.4)
    ws = weights(b)
    assert [y is not None for y in b] == list(z[f"{cid}/outputs"])
    sum((y * w).sum() for y, w in zip(b, ws) if y is not None).backward()
    assert [y.grad is not None for y in b_in] == list(z[f"{cid}/in_grads"])
    params = [(k, p.grad) for k, p in ours.named_parameters() if p.grad is not None]
    assert [k for k, _ in params] == str(z[f"{cid}/p_names"]).split("\n")
    assert len(params) >= 20
    # outputs and input gradients at fixed positions; parameter gradients at stored positions among the reference's
    # nonzero cells (a HexPlane gradient is nonzero only in the cells the 150 points touch)
    for name, ts, k in (("out", [y for y in b if y is not None], 64), ("in", [y.grad for y in b_in if y.grad is not None], 64)):
        refs = np.split(z[f"{cid}/{name}_s"], np.cumsum([min(t.numel(), k) for t in ts])[:-1])
        for i, (t, r) in enumerate(zip(ts, refs)):
            e = util.relerr_sampled(t, r, z[f"{cid}/{name}_max"][i], k)
            assert e < TOL, (name, i, e)
    cuts = np.cumsum(z[f"{cid}/p_n"])[:-1]
    for i, ((k, t), idx, r) in enumerate(zip(params, np.split(z[f"{cid}/p_idx"], cuts), np.split(z[f"{cid}/p_s"], cuts))):
        ours_s = t.reshape(-1)[torch.from_numpy(idx.astype(np.int64))].numpy().astype(np.float64)
        e = float(np.abs(ours_s - r).max() / (z[f"{cid}/p_max"][i] + 1e-30)) if idx.size else 0.0
        assert e < TOL, (k, e)


def test_unrunnable_upstream_switches_raise_with_the_reason():
    from s3gaussian_b200.deformation import deform_network
    for flag in (dict(no_grid=True), dict(grid_pe=2)):
        with pytest.raises(NotImplementedError, match="reference"):
            deform_network(ref_ext.ref_deform_args((16, 12, 10, 7), (1, 2), **flag))
