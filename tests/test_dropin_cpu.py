"""Host-side half of the drop-in proof (no GPU): after `sparf_b200.install_as_reference_renderer()` a trainer module that
imports `Graph` from `source.models.renderer` and subclasses it, as the reference's `joint_pose_nerf_trainer.py` does
(`from source.models.renderer import Graph` ... `class Graph(Graph):`), derives from OUR `Graph`.  The GPU half (our
renderer and loss modules against the goldens the reference produced) is tests/test_losses.py::test_full_sparf_step_vs_reference."""
import sys
import types

_SWAPPED = ("source.models.renderer", "source.models.frequency_nerf")

_TRAINER = """
from source.models.renderer import Graph


class Graph(Graph):
    pass
"""


def test_reference_trainer_graph_subclasses_our_graph():
    import sparf_b200
    import sparf_b200.frequency_nerf
    import sparf_b200.renderer
    saved = {k: sys.modules.get(k) for k in _SWAPPED}
    try:
        sparf_b200.install_as_reference_renderer()
        assert sys.modules["source.models.renderer"] is sparf_b200.renderer
        assert sys.modules["source.models.frequency_nerf"] is sparf_b200.frequency_nerf
        trainer = types.ModuleType("source.training.joint_pose_nerf_trainer")
        exec(compile(_TRAINER, trainer.__name__, "exec"), trainer.__dict__)
        assert sparf_b200.renderer.Graph in trainer.Graph.__mro__
        assert trainer.Graph is not sparf_b200.renderer.Graph
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
