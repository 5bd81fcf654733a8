"""GPU test: the Python surface object for object against the unmodified reference's own module (oracle/_ref/cityflow*.so,
through its pinned transcript): tests/api_parity_main.py with the real `cityflow` drop-in.  The CPU suite runs the same
comparison with the module linked over the emulated device.  (Sorted last: added after the round's last GPU session.)"""
import pytest

pytestmark = pytest.mark.gpu


def test_python_surface_object_for_object_vs_reference_module(cfg_6x6_rl):
    import cityflow
    import api_parity_main
    stats = api_parity_main.compare_with_reference(cityflow, cfg_6x6_rl, 520)
    assert stats["infos"] > 2000 and stats["custom"] > 80 and stats["rerouted_ok"] > 10 and stats["vehicles"] > 500
