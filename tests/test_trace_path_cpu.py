"""CPU: which traces run the wavefront path (workspace for live rays, host round trips, no CUDA-graph capture)."""
import optable_b200 as ob
from optable_b200.backend import Engine, runs_wavefront
from optable_b200.flatten import FlatScene
from tests import scenes


def _flat(sc):
    return FlatScene(sc.components, sc.monitors)


def test_runs_wavefront():
    plain = _flat(scenes.mirror_pair(ob))
    assert plain.max_children == 1 and not plain.n_capslots and not plain.has_pass
    prm = Engine.make_params
    assert not runs_wavefront([plain], prm())
    assert not runs_wavefront([plain, plain], prm())
    assert runs_wavefront([plain], prm(chain_len=4))
    assert runs_wavefront([plain], prm(flag_ambiguity=True))
    assert runs_wavefront([plain], prm(reference_roots=True))
    splitting = _flat(scenes.glass_slab(ob))
    assert splitting.max_children == 2 and runs_wavefront([splitting], prm())
    assert runs_wavefront([plain, splitting], prm())
    capped = FlatScene([ob.Mirror([0, 0, 0], max_interact_count=3)])
    assert capped.max_children == 1 and capped.n_capslots == 1 and runs_wavefront([capped], prm())
    passing = _flat(scenes.monitor_as_component(ob))
    assert passing.max_children == 1 and not passing.n_capslots and passing.has_pass
    assert runs_wavefront([passing], prm())
