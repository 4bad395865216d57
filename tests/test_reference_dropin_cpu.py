"""CPU dry run of tests/test_gpu_reference_dropin.py: the vector-store calls the reference's own operators made on FaissVS
(tests/golden/reference_vs_calls.*) are replayed on B200VS with the native index replaced by the oracle-backed fake. Checks
the host side the GPU test relies on (directory layout, argument types, id remapping, -1 padding); the numbers come from the
oracle here."""
from helpers import FakeIndex, replay_reference_vs_calls


def test_reference_vs_calls_replay_over_b200vs_host_logic(monkeypatch, tmp_path):
    from lotus_b200 import _native as nv
    from lotus_b200.vs import B200VS
    monkeypatch.setattr(nv, "Index", FakeIndex)
    monkeypatch.setattr(nv, "require_device", lambda: None)
    vs = B200VS(dtype="f32")
    assert replay_reference_vs_calls(vs, str(tmp_path)) > 0
    vs.close()
