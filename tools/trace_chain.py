#!/usr/bin/env python
"""Wait-time breakdown of the warp roles of the tcgen05 chain kernels.

Needs the tracing library, built by `python -m sparf_b200.build --trace` and loaded with
SPARF_B200_LIB=sparf_b200/lib/libsparf_b200_trace.so (the kernels then accumulate, per role, the clocks spent in each
mbarrier wait and print the mean over CTAs to stderr after every launch).  Debug tool, not part of the product.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    sys.path.insert(0, p)
import torch

import common
from sparf_b200 import _lib, ops


def main():
    R, S = 1023, 128
    opt = common.make_opt(S=S)
    sd = common.det_weights(opt, 0)
    keys = sum([["mlp_feat.%d.weight" % i, "mlp_feat.%d.bias" % i] for i in range(8)], []) + \
        ["mlp_rgb.0.weight", "mlp_rgb.0.bias", "mlp_rgb.1.weight", "mlp_rgb.1.bias"]
    params = [sd[k].cuda().requires_grad_(True) for k in keys]
    o = torch.randn(R, 3, device="cuda") * 0.3
    d = torch.nn.functional.normalize(torch.randn(R, 3, device="cuda"), dim=-1)
    t = torch.sort(torch.rand(R, S, device="cuda") * 4 + 1.2, dim=1).values
    spec = ops.MLPSpec()
    gs, gc = torch.randn(R, S, device="cuda"), torch.randn(R, S, 3, device="cuda")
    for eng in (_lib.ENGINE_TC_3X, _lib.ENGINE_TC_1X):
        for rep in range(2):
            sys.stderr.write("--- engine %d inference forward, rep %d\n" % (eng, rep))
            with torch.no_grad():
                ops.mlp_forward(spec, o, d, t, params, engine=eng)
            torch.cuda.synchronize()
    for rep in range(2):
        sys.stderr.write("--- training step (tape), rep %d\n" % rep)
        s, c = ops.mlp_forward(spec, o, d, t, params, engine=_lib.ENGINE_TC_3X)
        torch.autograd.backward([s, c], [gs, gc])
        torch.cuda.synchronize()


if __name__ == "__main__":
    main()
