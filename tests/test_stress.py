"""Cold-L2 repetitions of the taped MLP training step (tools/stress_chain.py): every repetition must reproduce the
first one bit-exactly in the forward outputs.  This is the test that exposes mbarrier protocol races between the warp
roles of the chain kernels (a lapped waiter hung one step in ~50 before the ring barriers counted every waiter)."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_cold_l2_repetitions_are_reproducible(monkeypatch, capsys):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import stress_chain
    monkeypatch.setattr(sys, "argv", ["stress_chain.py", "40"])
    stress_chain.main()
    assert "stress ok: 40 repetitions" in capsys.readouterr().out


# the recompute backward (its bf16 forward runs the shared-memory-operand chain kernel), plus a batch larger than one
# backward chunk (chunked tape walk with accumulating gradients); subprocesses, one per variant
VARIANTS = [
    ("recompute backward (no tape)", {"STRESS_TAPE": "0"}, ["25"]),
    ("two backward chunks", {}, ["15", "1100", "128"]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("what,env,argv", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_cold_l2_stress_of_selectable_variants(what, env, argv):
    import subprocess
    e = dict(os.environ)
    e.update(env)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stress_chain.py")] + argv, env=e, capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0 and "stress ok: %s repetitions" % argv[0] in res.stdout, (what, res.stdout[-500:], res.stderr[-1500:])
