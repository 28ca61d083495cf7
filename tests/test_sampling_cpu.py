"""RaySamplingStrategy / sample_rays mirrors (sparf_b200/sampling_strategies.py) against the reference's own classes:
same pools, same torch.randperm draws in the same order => identical rays under one seed.  The rays the reference drew
on the inputs below are stored in golden/reference_modules.npz (tests/golden/make_module_golden.py regenerates it)."""
import os

import numpy as np
import pytest
import torch

import common

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_modules.npz")
CASES = [dict(), dict(sampled_fraction_in_center=0.25), dict(depth_patch=0), dict(depth_patch=0, sampled_fraction_in_center=0.5)]
SAMPLE_RAYS_KW = [dict(nbr=50), dict(nbr=64, fraction_in_center=0.25), dict()]


def _opt(**kw):
    opt = common.make_opt(rand_rays=96)
    opt.sample_fraction_in_fg_mask = 0.0
    opt.sampled_fraction_in_center = 0.0
    opt.depth_regu_patch_size = 2
    for k, v in kw.items():
        if k == "depth_patch":
            opt.loss_weight.depth_patch = v
        else:
            opt[k] = v
    return opt


def ray_sampling_run(strategy_cls, sample_rays, case):
    """Rays drawn by `strategy_cls` (a RaySamplingStrategy) and by `sample_rays` under fixed seeds."""
    opt = _opt(**case)
    data = common.make_scene(3, 3, 24, 32)
    strategy = strategy_cls(opt, data_dict=data, device=torch.device("cpu"))
    out = {}
    for center in (False, True):
        torch.manual_seed(5)
        out["strategy_center%d" % center] = strategy(96, sample_in_center=center)
    for i, kw in enumerate(SAMPLE_RAYS_KW):
        torch.manual_seed(9)
        out["sample_rays%d_pixels" % i], out["sample_rays%d_rays" % i] = sample_rays(24, 32, **kw)
    return out


def sampling_golden_key(case_index, name):
    return "sampling_case%d_%s" % (case_index, name)


@pytest.mark.parametrize("case", CASES)
def test_ray_sampling_strategy_matches_reference(case):
    from sparf_b200.sampling_strategies import RaySamplingStrategy, sample_rays
    gold = np.load(GOLDEN)
    ours = ray_sampling_run(RaySamplingStrategy, sample_rays, case)
    for name, a in ours.items():
        b = torch.from_numpy(gold[sampling_golden_key(CASES.index(case), name)])
        assert a.shape == b.shape and torch.equal(a, b), name
