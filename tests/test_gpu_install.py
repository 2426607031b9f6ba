"""GPU: the literal drop-in. `optable_b200.install(reference)` swaps `OpticalTable.ray_tracing` of the UNMODIFIED
reference package (the `pip install --target baseline/_ref` copy that travels with the snapshot, SURVEY 8c) for the
CUDA engine; the same scene, built twice from the reference's OWN classes, is traced once by the reference's
original method on the host and once through liboptb.so, and compared object by object:
`table.rays`, `Monitor._data_raw`, `_interact_count`, the monitors' accessors, `calculate_abcd_matrix`
(/root/reference/optable/optical_table.py:57-147, 211-297)."""
import numpy as np
import pytest

from oracle import ref_harness as RH
from tests import parity, scenes
from tests.install_check import check_against_golden, check_install

pytestmark = pytest.mark.gpu


def _engine():
    from optable_b200.backend import Engine

    return Engine.get(0)


def _q_rtol(name):
    """q after an ASphere surface: the reference's finite-difference curvature amplifies rounding (SURVEY A.11)."""
    from optable_b200.flatten import FlatScene
    import optable_b200 as ob

    sc = scenes.REGISTRY[name](ob)
    return parity.q_rtol_for(sc.flat())


@pytest.mark.parametrize("name", sorted(scenes.REGISTRY))
def test_cuda_engine_under_reference_classes(name):
    """With the reference package installed: `optable_b200.install(reference)` swaps the CUDA engine into the
    reference's own `OpticalTable.ray_tracing`, and the scene built from the reference's classes is compared object
    by object with the reference's original method (tests/install_check.check_install). Without it: this package's
    own classes on the CUDA engine against the reference's stored results for the scene (tests/golden/<name>.npz,
    check_against_golden): segments, families, monitor rows and interact counts."""
    if RH.reference_available():
        n_seg, n_rows = check_install(name, _engine(), q_rtol=_q_rtol(name))
    else:
        n_seg, n_rows = check_against_golden(name, q_rtol=_q_rtol(name))
    assert n_seg > 0


def test_reference_abcd_matrix_on_cuda_backend(monkeypatch):
    """The reference's OWN `calculate_abcd_matrix` (three `ray_tracing` calls, monitor accessors sorted by ray id,
    optical_table.py:211-297) running on top of the swapped back end equals itself on the original back end.
    Without the reference package: _abcd_matrix_cuda_equals_oracle."""
    import optable_b200

    if not RH.reference_available():
        _abcd_matrix_cuda_equals_oracle(monkeypatch)
        return
    ref = RH.load_reference()

    def build():
        F1 = F2 = 43.17
        lens = scenes.asphere_lens9(ref, [F1, 0, 0])
        l1 = scenes.asphere_lens9(ref, [F1 + 2 * F2, 0, 0]).RotZ(np.pi)
        m0, m1 = ref.Monitor([0, 0, 0], width=5, height=5), ref.Monitor([2 * F1 + 2 * F2, 0, 0], width=5, height=5)
        t = ref.OpticalTable()
        t.add_components([lens, l1])
        t.add_monitors([m0, m1])
        return t, m0, m1

    ta, a0, a1 = build()
    want = ta.calculate_abcd_matrix(a0, a1, scenes.abcd_rays(ref))
    tb, b0, b1 = build()
    original = optable_b200.install(ref, engine=_engine())
    try:
        got = tb.calculate_abcd_matrix(b0, b1, scenes.abcd_rays(ref))
    finally:
        ref.OpticalTable.ray_tracing = original
    # finite differences of traced positions over 1e-5: 1e-9 trace parity -> ~1e-4 absolute on the entries
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=2e-4)
    assert len(ta.rays) == len(tb.rays) and len(a1._data_raw) == len(b1._data_raw)
    np.testing.assert_allclose(b1.get_yList(sort="ID"), a1.get_yList(sort="ID"), rtol=1e-9, atol=1e-12)


def _abcd_matrix_cuda_equals_oracle(monkeypatch):
    """The same 4f relay and call on this package's classes: `calculate_abcd_matrix` on the CUDA back end equals
    itself on the C restatement of the reference's loop (the oracle, checked against every stored reference result
    in tests/test_oracle_golden.py). tests/test_gpu_api.py checks the matrices of a different relay against the
    reference's stored values; this keeps the back-end swap of the live test, on its own geometry."""
    import optable_b200 as ob
    from optable_b200 import backend
    from tests.test_install_cpu import OracleEngine

    def build():
        F1 = F2 = 43.17
        lens = scenes.asphere_lens9(ob, [F1, 0, 0])
        l1 = scenes.asphere_lens9(ob, [F1 + 2 * F2, 0, 0]).RotZ(np.pi)
        m0, m1 = ob.Monitor([0, 0, 0], width=5, height=5), ob.Monitor([2 * F1 + 2 * F2, 0, 0], width=5, height=5)
        t = ob.OpticalTable()
        t.add_components([lens, l1])
        t.add_monitors([m0, m1])
        return t, m0, m1

    tb, b0, b1 = build()
    got = tb.calculate_abcd_matrix(b0, b1, scenes.abcd_rays(ob))      # liboptb.so
    monkeypatch.setattr(backend.Engine, "get", classmethod(lambda cls, device=None: OracleEngine()))
    ta, a0, a1 = build()
    want = ta.calculate_abcd_matrix(a0, a1, scenes.abcd_rays(ob))     # the C restatement on the host
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=2e-4)
    assert len(ta.rays) == len(tb.rays) and a1.ndata == b1.ndata > 0
    np.testing.assert_allclose(b1.get_yList(sort="ID"), a1.get_yList(sort="ID"), rtol=1e-9, atol=1e-12)


def test_native_library_is_what_ran():
    """The swapped method must run liboptb.so (no CPU path exists): the engine is the ctypes-bound CUDA context."""
    from optable_b200 import backend

    eng = _engine()
    assert isinstance(eng, backend.Engine) and backend.lib().optb_abi_version() > 0
    import ctypes

    maps = open("/proc/self/maps").read()
    assert "liboptb.so" in maps
