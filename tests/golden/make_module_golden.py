#!/usr/bin/env python
"""Generate tests/golden/reference_modules.npz by running the UNMODIFIED reference's pose-parameter and ray-sampling
modules on the inputs of tests/test_pose_models_cpu.py and tests/test_sampling_cpu.py:

    python tests/golden/make_module_golden.py <path of a SPARF checkout>

The tests build the same inputs, run this package's mirrors on them and compare with what is stored here.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main(reference_root):
    tests = os.path.dirname(HERE)
    for p in (os.path.dirname(tests), tests, HERE, os.path.join(HERE, "_shims"), reference_root):
        sys.path.insert(0, p)
    import numpy as np
    from source.models.poses_models.quaternion import QuaternionsPoseParameters
    from source.training.core import sampling_strategies

    import test_pose_models_cpu as P
    import test_sampling_cpu as S

    out = {}
    for case in P.REFERENCE_CASES:
        for name, v in P.quaternion_pose_run(QuaternionsPoseParameters, *case).items():
            out[P.pose_golden_key(*case, name)] = v.numpy()
    for i, case in enumerate(S.CASES):
        for name, v in S.ray_sampling_run(sampling_strategies.RaySamplingStrategy, sampling_strategies.sample_rays,
                                          case).items():
            out[S.sampling_golden_key(i, name)] = v.numpy()
    path = os.path.join(HERE, "reference_modules.npz")
    np.savez_compressed(path, **out)
    print("wrote %s (%d arrays)" % (path, len(out)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
