#!/usr/bin/env python
"""Kernel timeline of ONE CUDA-graph replay of a bench step (default config c2): start offset, duration, stream and name
of every kernel (torch.profiler = CUPTI activity records, warm caches), and the idle time of the busiest stream between
them.  Usage: python tools/step_timeline.py [config] [engine]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    sys.path.insert(0, p)
import torch
from torch.profiler import ProfilerActivity, profile


def main():
    import bench
    import sparf_b200
    from sparf_b200.distributed import FlatGradients
    from sparf_b200.graphs import GraphedStep
    cfg_name = sys.argv[1] if len(sys.argv) > 1 else "c2"
    sparf_b200.set_engine(sys.argv[2] if len(sys.argv) > 2 else "auto")
    dev = torch.device("cuda")
    cfg = bench.CONFIGS[cfg_name]
    pr = bench.build_problem(cfg_name, dev, seed=0)
    pr.net.device_side_rng = True
    pr.loss_module.check_finite = False
    fg = FlatGradients(pr.modules)
    idx = torch.randperm(cfg["H"] * cfg["W"])[:cfg["rand_rays"] // cfg["B"]].to(dev)

    def step(i):
        fg.flat.zero_()
        return pr.forward_backward(i)

    step(idx)
    g = GraphedStep(step, (idx,), warmup=2)
    for _ in range(5):
        g(idx)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g(idx)
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type.name == "CUDA"]
    evs.sort(key=lambda e: e.time_range.start)
    t0 = evs[0].time_range.start
    end = max(e.time_range.end for e in evs)
    print("config %s: %d kernels / copies, %.1f us from the first start to the last end" % (cfg_name, len(evs), end - t0))
    last_end = t0
    for e in evs:
        gap = e.time_range.start - last_end
        print("%9.1f us  +%7.1f us  gap %6.1f  %s" % (e.time_range.start - t0, e.time_range.end - e.time_range.start,
                                                     gap if gap > 0 else 0.0, e.name[:100]))
        last_end = max(last_end, e.time_range.end)


if __name__ == "__main__":
    main()
