"""GPU test of the archive in the reference's JSON schema (SURVEY.md section 8 row f2): Archive.dump("x.json") and
load_from_file() interchange with the unmodified reference (oracle/_ref/refdump `archive` / `resume`, pinned) in both
directions.
The checks (tests/archive_checks.py), the host logic and the image codec are the ones tests/test_cpu.py runs over the
emulated device; here the image goes to / comes from the real device through DeviceSim::snapshotToHost /
snapshotFromHost + restore, the calls the binary archive uses.

(Sorted last on purpose: this path was written after the last GPU session of its round, so under `pytest -x` a surprise
here cannot hide the results of the parity suites.)"""
import json

import pytest

import archive_checks

pytestmark = pytest.mark.gpu


def _engine(cfg):
    from cityflow_b200.capi import CEngine
    return CEngine(cfg)


def test_json_archive_interchanges_with_the_reference(cfg_3x3_dense, tmp_path):
    archive_checks.check_json_interchange(_engine, cfg_3x3_dense, str(tmp_path))


def test_json_archive_with_rl_phases(cfg_6x6_rl, tmp_path):
    archive_checks.check_json_with_rl_phases(_engine, cfg_6x6_rl, str(tmp_path))


def test_json_archive_through_the_python_module(cfg_3x3_dense, tmp_path):
    """The drop-in module, as the reference's tests/python/test_archive.py:99-102 uses it: snapshot().dump("save.json"),
    load_from_file("save.json")."""
    import cityflow
    eng = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    for _ in range(80):
        eng.next_step()
    path = str(tmp_path / "save.json")
    eng.snapshot().dump(path)
    doc = json.load(open(path))
    assert doc["step"] == 80 and doc["activeVehicleCount"] == eng.get_vehicle_count()
    assert len(doc["vehicles"]) == len(eng.get_vehicles(include_waiting=True))
    eng2 = cityflow.Engine(cfg_3x3_dense, thread_num=1)
    eng2.load_from_file(path)
    assert eng2.get_current_time() == 80.0 and eng2.get_vehicle_count() == eng.get_vehicle_count()
    assert sorted(eng2.get_vehicles(include_waiting=True)) == sorted(eng.get_vehicles(include_waiting=True))
    assert eng2.get_lane_vehicle_count() == eng.get_lane_vehicle_count()


def test_reference_disk_io_archive_tests(cfg_6x6, tmp_path):
    """tests/python/test_archive.py:95-119 of the reference through the drop-in module, "save.json" and all."""
    import cityflow

    class Eng:
        def __init__(self, cfg):
            self.e = cityflow.Engine(cfg, thread_num=4)

        def next_step(self, n=1):
            for _ in range(n):
                self.e.next_step()

        def dump(self, path):
            self.e.snapshot().dump(path)

        def load_from_file(self, path):
            self.e.load_from_file(path)

    archive_checks.check_reference_disk_io_tests(Eng, cfg_6x6, str(tmp_path),
                                                 lambda x: (x.e.get_lane_vehicle_count(), x.e.get_average_travel_time()))


def test_lane_change_snapshot(tmp_path):
    """snapshot / dump / load_from_file with laneChange = true: the per-vehicle lane-change state travels in the image."""
    from cityflow_b200 import scenario
    cfg = scenario.make_grid_scenario(str(tmp_path), 3, 3, dense=dict(frac=1.0, interval=3.0, seed=3), name="s33lc", lane_change=True)
    archive_checks.check_lane_change_snapshot(_engine, cfg, str(tmp_path))
