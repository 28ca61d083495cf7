"""Pose-parameter modules vs the reference's own modules.  What the reference's QuaternionsPoseParameters computed on
the inputs below is stored in golden/reference_modules.npz (tests/golden/make_module_golden.py regenerates it)."""
import os

import numpy as np
import pytest
import torch

import common
from sparf_b200.poses_models import QuaternionsPoseParameters
from sparf_b200.utils.edict import edict

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_modules.npz")
REFERENCE_CASES = [(False, False, True, True), (True, True, True, True), (True, False, False, True), (False, True, True, False)]


def _opt(c2w, rel, rot=True, trans=True):
    opt = edict()
    opt.camera = edict(optimize_c2w=c2w, optimize_trans=trans, optimize_rot=rot, optimize_relative_poses=rel,
                       n_first_fixed_poses=1)
    return opt


def _poses(seed, n=4):
    data = common.make_scene(seed, n, 24, 32)
    return common.perturb_poses(data.pose, seed)


@pytest.mark.parametrize("c2w", [False, True])
@pytest.mark.parametrize("rel", [False, True])
def test_quaternion_pose_model_round_trip_and_gradients(c2w, rel):
    w2c = _poses(3)
    m = QuaternionsPoseParameters(_opt(c2w, rel), 4, w2c, torch.device("cpu"))
    assert torch.allclose(m.get_w2c_poses(), w2c, atol=2e-6)
    assert m.rot_embedding.shape == (4 - (1 if rel else 0), 4)
    loss = (m.get_w2c_poses() * torch.linspace(-1, 1, 48).view(4, 3, 4)).sum()
    loss.backward()
    assert m.rot_embedding.grad.abs().sum() > 0 and m.trans_embedding.grad.abs().sum() > 0


def quaternion_pose_run(cls, c2w, rel, rot, trans):
    """Build a pose model of class `cls`, move it off its initial value, and return what it computes."""
    w2c = _poses(5)
    m = cls(_opt(c2w, rel, rot, trans), 4, w2c, torch.device("cpu"))
    out = dict(rot_embedding=torch.as_tensor(m.rot_embedding).detach().clone())
    with torch.no_grad():       # move off the initial value the same way for every implementation
        if rot:
            m.rot_embedding += 0.05 * torch.arange(m.rot_embedding.numel()).view_as(m.rot_embedding).float().cos()
        if trans:
            m.trans_embedding += 0.1
    out["w2c"] = m.get_w2c_poses().detach()
    out["c2w"] = m.get_c2w_poses().detach()
    return out


def pose_golden_key(c2w, rel, rot, trans, name):
    return "quaternion_%d%d%d%d_%s" % (c2w, rel, rot, trans, name)


@pytest.mark.parametrize("c2w,rel,rot,trans", REFERENCE_CASES)
def test_quaternion_pose_model_matches_reference_module(c2w, rel, rot, trans):
    gold = np.load(GOLDEN)
    ours = quaternion_pose_run(QuaternionsPoseParameters, c2w, rel, rot, trans)
    for name in ("rot_embedding", "w2c", "c2w"):
        ref = torch.from_numpy(gold[pose_golden_key(c2w, rel, rot, trans, name)])
        assert ours[name].shape == ref.shape and torch.allclose(ours[name], ref, atol=1e-6), name
